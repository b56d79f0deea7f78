/* b3d — C-ABI of the B200-native hot path of vliu15/3d-brain-tumor-segmentation.
 *
 * The reference has no FFI of its own: its "operator API" is the Keras layer surface
 * (layers/*.py, model.py, util.py).  Each entry point below is the arithmetic behind one of
 * those call sites (cited as reference file:line) and is what the Python layer classes in
 * `3d-brain-tumor-segmentation_b200/` bind through ctypes (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *  - every tensor argument is a BORROWED `const DLTensor*` (include/b3d_dlpack.h); a
 *    `DLManagedTensor*` from `to_dlpack` may be passed as-is.  The callee never frees, never
 *    retains past return (+ stream order); outputs and workspaces are caller-allocated.  NULL is
 *    allowed only where marked "nullable".  The ONE allocation the library makes itself is a 64 MB
 *    split-K workspace per device, created on the first convolution call that wants it (never
 *    while the stream is capturing) and shared by all streams of that device: convolution calls
 *    on one device must therefore be ordered with respect to each other (one compute stream per
 *    device — the execution model of DESIGN.md section 5).
 *  - tensors must live on a CUDA device (kDLCUDA) — there is NO CPU path — and be fp32 unless
 *    stated otherwise; activations are channels_last [B, D, H, W, C], compact row-major
 *    (conv inputs/outputs may be channel slices of a wider NDHWC buffer); weights use the Keras
 *    layouts: Conv3D (kd,kh,kw,Cin,Cout), Conv3DTranspose (kd,kh,kw,Cout,Cin), Dense (in,out).
 *  - `void* stream` is a cudaStream_t; all work is enqueued on it, nothing synchronises, so
 *    every call is CUDA-graph capturable.
 *  - return 0 on success, a negative B3D_ERR_* code otherwise; `b3d_last_error()` returns the
 *    thread-local message.  No exceptions cross the ABI.  Process-wide state is limited to the
 *    settings below (b3d_set_conv_precision, b3d_set_conv_kdfold, b3d_set_wgrad_ts) and the split-K workspace.
 */
#ifndef B3D_H_
#define B3D_H_
#include "b3d_dlpack.h"

#ifdef __cplusplus
extern "C" {
#endif

#define B3D_ERR_ARG (-1)
#define B3D_ERR_DEVICE (-2)
#define B3D_ERR_DTYPE (-3)
#define B3D_ERR_LAYOUT (-4)
#define B3D_ERR_SHAPE (-5)
#define B3D_ERR_CUDA (-6)
#define B3D_ERR_UNSUPPORTED (-7)

const char* b3d_last_error(void);
int b3d_abi_version(void);

/* ---- Conv3D / Conv3DTranspose, TF 'same' padding ------------------------------------------
 * replaces tf.keras.layers.Conv3D at resnet.py:30-37 (1x1x1), :64-73, :80-87, :96-103 (3x3x3),
 * downsample.py:28-35 (k3 s2: pad_before 0 / pad_after 1), decoder.py:55-63 (1x1x1 + sigmoid),
 * vae.py:92-99, and tf.keras.layers.Conv3DTranspose at upsample.py:28-33 (k3 s2 = adjoint of the
 * strided SAME conv; output = 2x input).
 *   stride: 1, or 2 (k=3 only; even sizes).  transposed: 1 => Conv3DTranspose (stride must be 2).
 *   act: 0 none, 1 sigmoid.  accumulate: y += result.
 *   gn_stats (nullable): fp64 [B, groups, 2], receives (sum, sum of squares) of y per GroupNorm
 *     chunk straight from the conv epilogue.  gap (nullable): fp32 [B, Cout] = sum over voxels of y.
 *   wpacked (nullable): weights re-laid-out by b3d_conv3d_pack_weights => run the tcgen05
 *     implicit-GEMM kernel (requires b3d_conv3d_tc_supported); NULL => CUDA-core kernel. */
int b3d_conv3d_fwd(const DLTensor* x, const DLTensor* w, const DLTensor* bias /*nullable*/, DLTensor* y,
                   int stride, int transposed, int act, DLTensor* gn_stats, int groups, DLTensor* gap,
                   int accumulate, const DLTensor* wpacked, void* stream);
/* Depth-slab form for whole-volume inference sharded along D (test.py:133 on the padded [1,160,192,160,C] volume,
 * one slab per GPU): x carries halo_before / halo_after (0|1) extra depth slices — the neighbour slabs' boundary
 * slices, zeros at the ends of the volume — and y holds only this slab's slices, so that the concatenation of
 * the slabs' y equals the conv of the whole volume.  conv k3 s1: (1,1); conv k3 s2: (0,1); conv-transpose: (1,0). */
int b3d_conv3d_fwd_halo(const DLTensor* x, const DLTensor* w, const DLTensor* bias /*nullable*/, DLTensor* y,
                        int stride, int transposed, int act, int halo_before, int halo_after, DLTensor* gap,
                        const DLTensor* wpacked, void* stream);
/* data gradient (what tape.gradient computes for the layer input, train.py:151) */
int b3d_conv3d_dgrad(const DLTensor* dy, const DLTensor* w, DLTensor* dx, int stride, int transposed,
                     int accumulate, const DLTensor* wpacked, void* stream);
/* weight (+ bias, nullable) gradient.  x_bf16 / dy_bf16 (nullable, bf16): scratch buffers of
 * voxels * (channels per voxel reported by b3d_conv3d_wgrad_plan) elements; when both are given they are filled
 * with bf16 copies of x / dy (space-to-depth order for stride 2, all taps stacked for narrow tensors) and the
 * tcgen05 kernel (bf16 operands, fp32 accumulation) is used, else the fp32 CUDA-core kernel.
 * x_bf16_ready != 0: x_bf16 already holds the plain bf16 copy of x (stride-1 layers sharing their input). */
int b3d_conv3d_wgrad(const DLTensor* x, const DLTensor* dy, DLTensor* dw, DLTensor* dbias, int stride,
                     int transposed, const DLTensor* x_bf16, const DLTensor* dy_bf16, int x_bf16_ready,
                     void* stream);
int b3d_conv3d_wgrad_tc_supported(int k, int stride, int transposed, int cin, int cout);
/* narrow-output 3x3x3 layers (Cout <= 32) use the TS-mode kernel (A operand in tensor memory, csrc/conv_tc_wgrad_ts.cu)
 * unless switched off (A/B comparisons, tests) */
int b3d_set_wgrad_ts(int on);
/* returns 0 (CUDA cores), 1 (plain copies), 2 / 3 (narrow input / output: tap-stacked copy); *x_ch, *dy_ch
 * receive the bf16 channels per voxel of the two scratch buffers */
int b3d_conv3d_wgrad_plan(int k, int stride, int transposed, int cin, int cout, long long* x_ch, long long* dy_ch);
/* 1 when the tcgen05 kernel runs the forward (dgrad=0) / data-gradient (dgrad=1) pass of a layer whose Keras
 * kernel is (k,k,k,a,b): stride-1 k in {1,3}, and the k3 stride-2 family (Conv3D s2, Conv3DTranspose), which is
 * executed as a 2x2x2 stride-1 conv over the coarse grid with space-to-depth addressing (csrc/conv_s2.cu). */
int b3d_conv3d_tc_supported(int k, int stride, int transposed, int dgrad, int a, int b);
/* operand type of the tcgen05 conv MMAs (0 = tf32, 1 = bf16, 2 = fp16) for the forward pass and for the data
 * gradient; defaults: forward fp16 (TF32's 11-bit significand), backward bf16; fp32 accumulation either way.
 * Packed weights depend on it: re-pack after a change.  get: fwd | bwd << 4. */
int b3d_set_conv_precision(int fwd_op, int bwd_op);
int b3d_get_conv_precision(void);
/* kd-folded variant of the 3x3x3 tcgen05 kernel for output tiles of 16 / 32 channels (depth taps folded into the MMA
 * N dimension: 2-2.4x fewer small-N MMAs; csrc/conv_tc.cu).  Process-wide, default ON; changes the packed weight
 * layout of those layers (re-pack after switching).  Returns the previous setting. */
int b3d_set_conv_kdfold(int on);
long long b3d_conv3d_packed_elems(int k, int stride, int a, int b);
int b3d_conv3d_pack_weights(const DLTensor* w, DLTensor* packed, int stride, int transposed, int dgrad,
                            void* stream);
/* Batched re-layout, one launch for every layer of a model (run after the optimiser step; the reference has no
 * counterpart — Keras hands cuDNN the HWIO kernel every call).  b3d_conv3d_pack_job writes the table entry of one
 * layer/pass into `job_out` (host memory, b3d_conv3d_pack_job_bytes() bytes) with `block0` = the sum of *blocks of
 * the entries before it; the concatenated entries, uploaded as an int64 device tensor, drive b3d_conv3d_pack_many
 * (`blocks` = the total).  The entries hold the device pointers of w / packed: both must stay where they are. */
int b3d_conv3d_pack_job_bytes(void);
int b3d_conv3d_pack_job(const DLTensor* w, DLTensor* packed, int stride, int transposed, int dgrad,
                        long long block0, void* job_out, long long* blocks);
int b3d_conv3d_pack_many(const DLTensor* jobs /*int64 table*/, int njobs, long long blocks, void* stream);

/* ---- GroupNormalization.call, channels_last semantics (group_norm.py:83-124; SURVEY F1) -----
 * "group" g = g-th contiguous 1/G chunk of each sample's flat buffer; eps inside sqrt; population
 * variance.  stats: fp64 [B, G, 2] = (sum x, sum x^2).  relu=1 fuses the following Activation('relu')
 * (resnet.py:95,111; downsample.py:39; upsample.py:37).  Errors (B3D_ERR_SHAPE, reference
 * ValueError text) when C < groups or C % groups != 0 (group_norm.py:51-59).
 *   Window (stats, apply): total_vox = 0 => x is the whole tensor, any batch.  total_vox > 0 => x is the window
 *     [vox_offset, vox_offset + voxels of x) of a batch-1 volume of total_vox voxels (depth-slab inference; chunk
 *     boundaries need not coincide with the window's): gn_stats writes the window's PARTIAL (sum, sum^2) per chunk of
 *     the WHOLE volume (fp64 [1, G, 2]; the caller all-reduces them), gn_apply normalises the window with the reduced
 *     statistics.
 *   P16 twins (see "P16 operand twins" below): gn_apply with y16 (fp16 | bf16) given writes it, y16b (nullable) a
 *     second, bf16 twin for the weight gradient of the consuming conv, and y becomes nullable (NULL = twin only);
 *     needs C = 8 * 2^k and a cell-aligned window, else B3D_ERR_UNSUPPORTED / B3D_ERR_LAYOUT.  gn_bwd_apply with dx16
 *     (bf16) given writes the twin for the data / weight gradient of the conv that produced x, dx becomes nullable and
 *     dbias (nullable, fp32 [C]) receives the column sums of dx = that conv's bias gradient.  Without twins y / dx
 *     are required.  B3D_ERR_ARG: y16b without y16, dbias without dx16, neither dx nor dx16. */
int b3d_gn_stats(const DLTensor* x, DLTensor* stats, int groups, long long vox_offset, long long total_vox,
                 void* stream);
int b3d_gn_apply(const DLTensor* x, const DLTensor* stats, const DLTensor* gamma, const DLTensor* beta,
                 DLTensor* y /*nullable*/, DLTensor* y16 /*nullable*/, DLTensor* y16b /*nullable*/, int groups,
                 float eps, int relu, long long vox_offset, long long total_vox, void* stream);
int b3d_gn_bwd_reduce(const DLTensor* dy, const DLTensor* x, const DLTensor* stats, const DLTensor* gamma,
                      const DLTensor* beta, DLTensor* dgamma, DLTensor* dbeta, DLTensor* csum /*fp64 [B,G,2]*/,
                      int groups, float eps, int relu, void* stream);
int b3d_gn_bwd_apply(const DLTensor* dy, const DLTensor* x, const DLTensor* stats, const DLTensor* gamma,
                     const DLTensor* beta, const DLTensor* csum, DLTensor* dx /*nullable*/,
                     DLTensor* dx16 /*nullable*/, DLTensor* dbias /*nullable*/, int groups, float eps, int relu,
                     void* stream);

/* ---- GroupNormalization with TRUE channel groups — the reference's data_format='channels_first' semantics
 * (group_norm.py axis=1: group g = channels [g*C/G, (g+1)*C/G) of every voxel), on the same NDHWC storage
 * (csrc/norm_channel.cu).  stats / csum: fp64 [B, G, 2].  gn_channel_bwd runs the reduction pass (dgamma, dbeta,
 * csum) and the elementwise pass (dx).  relayout: NCDHW <-> NDHWC copies for the channels_first API surface. */
int b3d_gn_channel_stats(const DLTensor* x, DLTensor* stats, int groups, void* stream);
int b3d_gn_channel_apply(const DLTensor* x, const DLTensor* stats, const DLTensor* gamma, const DLTensor* beta,
                         DLTensor* y, int groups, float eps, int relu, void* stream);
int b3d_gn_channel_bwd(const DLTensor* dy, const DLTensor* x, const DLTensor* stats, const DLTensor* gamma,
                       const DLTensor* beta, DLTensor* dgamma, DLTensor* dbeta, DLTensor* csum, DLTensor* dx,
                       int groups, float eps, int relu, void* stream);
/* Depth-slab form (sharded inference, slab.py): x = one slab [1, Dl, H, W, C]; stats fp64 [1, G, 2] = the all-reduced
 * sums of every group over the whole volume of total_voxels voxels (the slabs' gn_channel_stats added up).  Writes the
 * fp32 y and / or the P16 twin y16 [1, Dl, H, C/8, W, 8] (fp16 or bf16); each is nullable, not both.  C % 8 == 0. */
int b3d_gn_channel_apply_slab(const DLTensor* x, const DLTensor* stats, const DLTensor* gamma, const DLTensor* beta,
                              DLTensor* y, DLTensor* y16, int groups, float eps, int relu, long long total_voxels,
                              void* stream);
int b3d_relayout(const DLTensor* src, DLTensor* dst, int to_channels_last, void* stream);

/* ---- ResnetBlock epilogue (resnet.py:121-137) --------------------------------------------------
 * chse = sigmoid(relu(gap_sum*inv_vox . W1) . W2);  out = res*(sigmoid(res.w_sp)+chse) + relu(GN2(h2)).
 * has_gn=0: h2 is already normalised+activated (stats/gamma/beta NULL).
 *   P16 twins (see "P16 operand twins" below): block_epilogue_fwd with out16 (fp16 | bf16) given writes it, out16b
 *     (nullable) a second, bf16 twin for the weight gradients of the consuming convs, and out becomes nullable (NULL =
 *     twin only).  Only then may it take a window: total_vox > 0 => res / h2 / out16 hold voxels [vox_offset,
 *     vox_offset + D*H*W) of a batch-1 volume of total_vox voxels, stats = the all-reduced GroupNorm statistics of the
 *     whole volume, chse from the all-reduced pooling sums; total_vox = 0 => the tensors are the whole volume.
 *     block_epilogue_bwd_apply with dres16 / dh216 (bf16) given (has_gn = 1 only) writes the twins for the data / weight
 *     gradients of the pointwise and the second 3x3x3 conv, dres / dh2 become nullable (each gradient needs its fp32
 *     output or its twin) and dbias_res / dbias_h2 (nullable, both or none, fp32 [F]) receive their column sums =
 *     those convs' bias gradients.  Without twins out, dres and (has_gn) dh2 are required.  The twin kernels need
 *     F = 8 * 2^k <= 256 (else B3D_ERR_UNSUPPORTED).  B3D_ERR_ARG: out16b without out16, bias gradients without a twin,
 *     a gradient with neither output. */
int b3d_se_fc_fwd(const DLTensor* gap_sum, const DLTensor* w1, const DLTensor* w2, DLTensor* hidden,
                  DLTensor* chse, float inv_vox, void* stream);
int b3d_se_fc_bwd(const DLTensor* gap_sum, const DLTensor* w1, const DLTensor* w2, const DLTensor* hidden,
                  const DLTensor* chse, const DLTensor* dchse, DLTensor* dw1, DLTensor* dw2, DLTensor* dgap,
                  float inv_vox, void* stream);
int b3d_block_epilogue_fwd(const DLTensor* res, const DLTensor* h2, const DLTensor* stats, const DLTensor* gamma,
                           const DLTensor* beta, const DLTensor* wsp, const DLTensor* chse, DLTensor* out /*nullable*/,
                           DLTensor* out16 /*nullable*/, DLTensor* out16b /*nullable*/, int groups, float eps,
                           int has_gn, long long vox_offset, long long total_vox, void* stream);
int b3d_block_epilogue_bwd_reduce(const DLTensor* dout, const DLTensor* res, const DLTensor* h2,
                                  const DLTensor* stats, const DLTensor* gamma, const DLTensor* beta,
                                  const DLTensor* wsp, DLTensor* dchse, DLTensor* dwsp, DLTensor* dgamma,
                                  DLTensor* dbeta, DLTensor* csum, int groups, float eps, int has_gn,
                                  void* stream);
int b3d_block_epilogue_bwd_apply(const DLTensor* dout, const DLTensor* res, const DLTensor* h2,
                                 const DLTensor* stats, const DLTensor* gamma, const DLTensor* beta,
                                 const DLTensor* wsp, const DLTensor* chse, const DLTensor* dgap,
                                 const DLTensor* csum, DLTensor* dres /*nullable*/, DLTensor* dh2 /*nullable*/,
                                 DLTensor* dres16 /*nullable*/, DLTensor* dh216 /*nullable*/,
                                 DLTensor* dbias_res /*nullable*/, DLTensor* dbias_h2 /*nullable*/, int groups,
                                 float eps, int has_gn, void* stream);

/* ---- VAE bottleneck (vae.py:9-13, :119-129): Dense, reparameterisation -------------------------*/
int b3d_dense_fwd(const DLTensor* x, const DLTensor* w, const DLTensor* bias, DLTensor* y, int act /*1 relu*/,
                  void* stream);
int b3d_dense_bwd(const DLTensor* x, const DLTensor* w, const DLTensor* y, const DLTensor* dy,
                  DLTensor* dx /*nullable*/, DLTensor* dw, DLTensor* db /*nullable*/, int act, void* stream);
int b3d_vae_sample_fwd(const DLTensor* proj /*[B,2L]=mean|logvar*/, const DLTensor* eps, DLTensor* z, void* stream);
int b3d_vae_sample_bwd(const DLTensor* proj, const DLTensor* eps, const DLTensor* dz, const DLTensor* dmean,
                       const DLTensor* dlogvar, DLTensor* dproj, void* stream);

/* ---- DiceVAELoss / DiceCoefficient (util.py:13-24, :35-57) --------------------------------------
 * sums: fp64 [3*C+2] workspace; out: fp32 [4] = total, dice, l2, kld.  y_vae NULL => dice only. */
int b3d_loss_fwd(const DLTensor* x, const DLTensor* y, const DLTensor* y_pred, const DLTensor* y_vae,
                 const DLTensor* z_mean, const DLTensor* z_logvar, DLTensor* sums, DLTensor* out, void* stream);
int b3d_loss_bwd(const DLTensor* x, const DLTensor* y, const DLTensor* y_pred, const DLTensor* y_vae,
                 const DLTensor* z_mean, const DLTensor* z_logvar, const DLTensor* sums, const DLTensor* gout,
                 DLTensor* dy_pred, DLTensor* dy_vae, DLTensor* dz_mean, DLTensor* dz_logvar, void* stream);
/* Batch-global objective under data parallelism (util.py:11,18-20 sums I, P, T over the BATCH axis too; SURVEY F6): each
 * rank runs b3d_loss_fwd on its crops, all-reduces (sum) the 3C+2 fp64 `sums` over the `replicas` ranks, calls
 * b3d_loss_finalize with the global element counts (out = the loss of the whole batch, identical on every rank) and
 * b3d_loss_bwd_dp for this rank's part of the gradient; the parameter gradients are then SUMMED over ranks, not averaged. */
int b3d_loss_finalize(const DLTensor* sums, DLTensor* out, long long n_rec_total, long long n_lat_total, void* stream);
int b3d_loss_bwd_dp(const DLTensor* x, const DLTensor* y, const DLTensor* y_pred, const DLTensor* y_vae,
                    const DLTensor* z_mean, const DLTensor* z_logvar, const DLTensor* sums, const DLTensor* gout,
                    DLTensor* dy_pred, DLTensor* dy_vae, DLTensor* dz_mean, DLTensor* dz_logvar, int replicas,
                    void* stream);
/* b3d_loss_fwd + b3d_dice_coeff of the same (y, y_pred) in ONE pass over them: the training loop evaluates both on the
 * same tensors (/root/reference/train.py:143,147; util.py:13-24, 35-57).  5-D NDHWC y / y_pred with W % 4 == 0. */
int b3d_loss_dice_fwd(const DLTensor* x, const DLTensor* y, const DLTensor* y_pred, const DLTensor* y_vae,
                      const DLTensor* z_mean, const DLTensor* z_logvar, DLTensor* sums, DLTensor* out,
                      DLTensor* acc /*fp32 [W*C*3]*/, DLTensor* dice /*fp32 [2]*/, int reduce_w, void* stream);
int b3d_dice_coeff(const DLTensor* y, const DLTensor* y_pred, DLTensor* acc /*fp32 [W*C*3]*/,
                   DLTensor* out /*fp32 [2] macro, micro*/, int reduce_w /*1: channels_first macro (util.py:36)*/,
                   void* stream);

/* ---- optimiser + regulariser (util.py:60-84 TF Adam, eps un-scaled; train.py:146 model.losses) ---*/
/* g_eff = g*grad_scale + decay*theta (first n_decay elements only; decay = 2*l2 in data-parallel mode) */
int b3d_adam_step(DLTensor* theta, DLTensor* m, DLTensor* v, const DLTensor* g,
                  DLTensor* state /*fp64 [2] = iterations, learning rate*/, float beta1, float beta2, float eps,
                  float grad_scale, float decay, long long n_decay, int tick, void* stream);
int b3d_l2_losses(const DLTensor* flat, const DLTensor* offsets /*int64 [n+1]*/, DLTensor* out /*[n]*/,
                  float scale, void* stream);
int b3d_l2_grad(const DLTensor* flat, DLTensor* grad, const DLTensor* offsets, const DLTensor* gout, float coef,
                void* stream);
int b3d_axpy(const DLTensor* flat, DLTensor* grad, long long n, float coef, const DLTensor* gout, void* stream);
/* out[0] = sum(v) + addend[0] (addend nullable): tf.reduce_sum(model.losses) added to the data loss,
 * /root/reference/train.py:146.  b3d_zero: cudaMemsetAsync of a contiguous fp32 tensor. */
int b3d_sum_add(const DLTensor* v, const DLTensor* addend /*nullable*/, DLTensor* out, void* stream);
int b3d_zero(DLTensor* t, void* stream);

/* ---- input Dropout (encoder.py:39,71), concat materialisation, small elementwise helpers --------*/
int b3d_dropout(const DLTensor* x, DLTensor* y, DLTensor* mask /*nullable*/, float rate, unsigned long long seed,
                DLTensor* counter /*int64 [1], nullable*/, void* stream);
int b3d_mul_scale(const DLTensor* a, const DLTensor* b, DLTensor* y, float scale, void* stream);
int b3d_sigmoid_bwd(const DLTensor* dy, const DLTensor* y, DLTensor* dx, void* stream);
int b3d_copy_channels(const DLTensor* src, DLTensor* dst, int accumulate, void* stream);

/* ---- training-example pipeline of tf.data's map function (train.py:12-47 parse_example) on the device ----------
 * channel_moments: x [D,H,W,C<=8] -> fp64 [C,2] (sum, sum of squares).  augment_crop: x += shift*sqrt(var); x *= scale
 * (train.py:20-24), crop window at (off_d, off_h, off_w) (train.py:27-28), flips of the crop (bit a = axis a,
 * train.py:31-35), labels y [D,H,W,1] -> one-hot without the background class (train.py:41-44).  The random draws
 * are the caller's. */
int b3d_channel_moments(const DLTensor* x, DLTensor* sums, void* stream);
int b3d_augment_crop(const DLTensor* x, const DLTensor* y, const DLTensor* sums, const DLTensor* shift,
                     const DLTensor* scale, DLTensor* x_out, DLTensor* y_out, int off_d, int off_h, int off_w,
                     int flip, void* stream);

/* ---- non-default resampling variants (csrc/resample.cu): MaxDownsample = MaxPooling3D(2, 2, 'same')
 * (downsample.py:51-70; even sizes, gradient to the first maximum of each window) and the UpSampling3D(size 2)
 * nearest-neighbour step of LinearUpsample (upsample.py:49-79).  NDHWC fp32, channels % 4 == 0. */
int b3d_maxpool2_fwd(const DLTensor* x, DLTensor* y, void* stream);
int b3d_maxpool2_bwd(const DLTensor* x, const DLTensor* dy, DLTensor* dx, void* stream);
int b3d_upsample2_fwd(const DLTensor* x, DLTensor* y, void* stream);
int b3d_upsample2_bwd(const DLTensor* dy, DLTensor* dx, void* stream);

/* ---- depth-slab sharded inference over NVLink peer memory (csrc/slab_comm.cu; host side slab.PeerComm) -----------
 * Every rank owns one symmetric buffer of b3d_slab_sym_bytes(mailbox_bytes) bytes mapped into its peers.
 * halo_exchange: my first / last boundary slices (send_prev / send_next, nullable) are stored into the neighbours'
 *   mailboxes and published with a system-scope release store; theirs are awaited (acquire spin on my own flags) and
 *   copied to recv_prev / recv_next (nullable).  prev_base / next_base: device addresses of the neighbours' symmetric
 *   buffers (0 = no neighbour).  epoch: int64 [1] device counter ticked once per forward (b3d_epoch_tick), seq: index
 *   of this exchange inside the forward.  peer_allreduce: in-place sum over all ranks (rank order, bit-identical
 *   everywhere) of <= 2 KB of fp32 / fp64 (GroupNorm chunk statistics, SE pooling sums); peer_allreduce2: a fp64 and a
 *   fp32 vector in one exchange. */
long long b3d_slab_sym_bytes(long long mailbox_bytes);
int b3d_halo_exchange(const DLTensor* send_prev, const DLTensor* send_next, DLTensor* recv_prev, DLTensor* recv_next,
                      long long prev_base, long long next_base, DLTensor* sym, const DLTensor* epoch, int seq,
                      long long mailbox_bytes, void* stream);
int b3d_peer_allreduce(DLTensor* x, const DLTensor* peers /*int64 [world]*/, int rank, DLTensor* sym,
                       const DLTensor* epoch, int seq, void* stream);
int b3d_peer_allreduce2(DLTensor* a /*fp64*/, DLTensor* b /*fp32*/, const DLTensor* peers, int rank, DLTensor* sym,
                        const DLTensor* epoch, int seq, void* stream);
int b3d_epoch_tick(DLTensor* epoch, void* stream);

/* Depth-slab form of the P16 forward conv (whole-volume inference sharded along D; /root/reference/test.py:133 on one
 * slab per GPU): the conv reads P16 sources that carry halo_before / halo_after extra depth slices and emits this slab's
 * PARTIAL GroupNorm statistics over the chunks of the whole volume (stat_total output voxels per sample, this slab's
 * first = stat_off; /root/reference/layers/group_norm.py:83-124 reshapes the whole volume); b3d_gn_apply and
 * b3d_block_epilogue_fwd take the all-reduced statistics and the same voxel window. */
int b3d_conv3d_fwd_p16_slab(const DLTensor* x0, const DLTensor* x1, const DLTensor* x2, const DLTensor* x3,
                            const DLTensor* w, const DLTensor* bias /*nullable*/, DLTensor* y, int stride,
                            int transposed, int act, int halo_before, int halo_after, DLTensor* gn_stats /*nullable*/,
                            int groups, long long stat_off, long long stat_total, DLTensor* gap /*nullable*/,
                            const DLTensor* wpacked, int prezeroed /*gn_stats / gap are already zero*/, void* stream);

/* ---- test-time augmentation (test.py:105-161): flip bits 1=D 2=H 4=W on one [D,H,W,C] volume ------------
 * flip_normalize: out = (flip(x) - mean)/std (test.py:107,128; mean/std nullable).
 * flip_accumulate: acc (+)= scale*flip(y), optionally multiplied by the brain mask (test.py:134,147-151). */
int b3d_flip_normalize(const DLTensor* x, const DLTensor* mean, const DLTensor* std, DLTensor* out, int flip,
                       void* stream);
int b3d_flip_accumulate(const DLTensor* y, DLTensor* acc, const DLTensor* mask, int flip, float scale, int first,
                        void* stream);

/* ---- evaluation of one segmented volume (csrc/metrics.cu; host side metrics.py) ------------------------------------
 * label_map: labels[d,h,w] = first argmax_c y_pred[d,h,w,c] + 1 where that maximum is > threshold, else 0 (the hard
 *   decision of b3d_dice_coeff); y_pred fp32 [D,H,W,C], C = 1..4; labels uint8 [d,h,w], d <= D, h <= H, w <= W (the
 *   leading corner: undoes pad_to_spatial_res).
 * region_surface: lut (uint8 [256]) maps a label to its region bits; counts (int64 [R,4], R <= 8) receives TP, FP, FN,
 *   TN per region; surf_pred / surf_true (uint8 [D,H,W]) get bit r where the voxel belongs to region r and has a
 *   6-neighbour outside it (outside the volume counts as outside).
 * surface_edt: edt (fp32 [R,D,H,W]) = squared Euclidean distance, with voxel spacing (sd, sh, sw), from every voxel to
 *   the nearest voxel with bit r of surf set; +inf where there is none.  Exact with unit spacing.  Lines up to 1024
 *   voxels on every axis.
 * hd95: out (fp64 [R,4]) = dice, sensitivity, specificity and the 95th percentile (numpy 'linear') of the distances from
 *   the prediction's surface to the truth's and back; 0 when both surfaces are empty, +inf when one is.  A ratio with a
 *   zero denominator is 1.  workspace: uint8, 16-byte aligned, >= 4 * R * (264 + 2 * D * H * W) bytes.
 * Each call clears what it accumulates; none allocates or synchronises, so the sequence can be graph-captured. */
int b3d_label_map(const DLTensor* y_pred, DLTensor* labels, float threshold, void* stream);
int b3d_region_surface(const DLTensor* pred, const DLTensor* true_labels, const DLTensor* lut, DLTensor* counts,
                       DLTensor* surf_pred, DLTensor* surf_true, void* stream);
int b3d_surface_edt(const DLTensor* surf, DLTensor* edt, int R, float sd, float sh, float sw, void* stream);
int b3d_hd95(const DLTensor* edt_true, const DLTensor* surf_pred, const DLTensor* edt_pred, const DLTensor* surf_true,
             const DLTensor* counts, DLTensor* out, DLTensor* workspace, void* stream);

/* ---- P16 operand twins -------------------------------------------------------------------------------------------
 * A "P16" tensor is the 16-bit copy of an activation (fp16) or gradient (bf16) in the layout the tcgen05 conv kernels
 * consume directly: [B, D, H, C/8, W, 8] (DLPack ndim 6, dtype f16 | bf16, compact).  Channel octets are planes inside
 * every (d, h) row: a voxel's 8 channels are one 16-byte UMMA cell and a halo row of one plane is W*16 contiguous bytes,
 * so whole halos are fetched as wide TMA rows.  The twins are written by the kernels that PRODUCE conv operands (the
 * twin outputs of b3d_gn_apply / b3d_block_epilogue_fwd and their backward-apply passes) — there is no cast pass on the
 * training step, and a channel concatenation (encoder.py:85,91; decoder.py:75) is a list of up to 4 sources. */
int b3d_p16_pack(const DLTensor* x /*fp32 NDHWC, C % 8 == 0, may be a channel slice*/, DLTensor* dst /*P16*/,
                 DLTensor* colsum /*nullable fp32 [C]: per-channel sums of x*/, void* stream);
int b3d_p16_unpack(const DLTensor* src /*P16*/, DLTensor* y /*fp32 NDHWC, may be a channel slice*/, void* stream);
int b3d_p16_copy_planes(const DLTensor* src /*P16*/, DLTensor* dst /*P16, wider*/, int c8off, void* stream);
int b3d_colsum(const DLTensor* x /*fp32 NDHWC*/, DLTensor* out /*fp32 [C]*/, void* stream);
/* The encoder's dense connections feed a block [a_last, a_0, .., a_last] (encoder.py:83-87: `inputs is cache[-1]`): the conv
 * over it equals a conv over [a_0, .., a_last] with the two weight slices of a_last added.  w: Keras kernel
 * (k,k,k,Cf+F,Cout); wf: its folded form (k,k,k,Cf,Cout); unfold scatters d(wf) back to d(w) (both slices of a_last get
 * the same gradient). */
int b3d_fold_dup(const DLTensor* w, DLTensor* wf, int F, void* stream);
int b3d_unfold_dup(const DLTensor* dwf, DLTensor* dw, int F, void* stream);
/* the three conv passes with P16 input operands (same semantics as b3d_conv3d_fwd / _dgrad / _wgrad; tcgen05 path only:
 * wpacked is required).  x0..x3: the sources whose channels are concatenated (x1..x3 nullable), all of the pass's MMA
 * operand type (forward: fp16 by default; data gradient: bf16).  The weight gradient takes bf16 twins of BOTH operands
 * (tcgen05 kind::f16 has one operand type for A and B; mixing f16 with bf16 is an illegal instruction), which is why
 * forward activations carry a second, bf16 twin (y16b / out16b above) when the forward type is fp16.  The weight gradient does NOT produce the bias gradient on this path: it is emitted
 * by the kernel that writes dy (`dbias` of b3d_gn_bwd_apply / b3d_block_epilogue_bwd_apply, `colsum` of
 * b3d_p16_pack).  scratch (nullable, 16-bit, 1-D): see b3d_conv3d_wgrad_p16_plan. */
int b3d_conv3d_fwd_p16(const DLTensor* x0, const DLTensor* x1, const DLTensor* x2, const DLTensor* x3, const DLTensor* w,
                       const DLTensor* bias /*nullable*/, DLTensor* y, int stride, int transposed, int act,
                       DLTensor* gn_stats, int groups, DLTensor* gap, int accumulate, const DLTensor* wpacked,
                       void* stream);
int b3d_conv3d_dgrad_p16(const DLTensor* dy /*P16*/, const DLTensor* w, DLTensor* dx, int stride, int transposed,
                         int accumulate, const DLTensor* wpacked, void* stream);
/* the same for a stride-1 conv whose input was a virtual channel concat: one compact dx tensor per concatenated piece */
int b3d_conv3d_dgrad_p16_split(const DLTensor* dy /*P16*/, const DLTensor* w, DLTensor* dx0, DLTensor* dx1 /*nullable*/,
                               DLTensor* dx2 /*nullable*/, DLTensor* dx3 /*nullable*/, int accumulate,
                               const DLTensor* wpacked, void* stream);
/* data gradient w.r.t. the input of a ResnetBlock from both convs reading it (/root/reference/layers/resnet.py:118,133):
 * dres (gradient of the pointwise conv's output) joins dy as a K segment used at the centre tap only */
int b3d_conv3d_dgrad_p16_block(const DLTensor* dy /*P16*/, const DLTensor* dres /*P16*/, const DLTensor* w,
                               const DLTensor* w_pw, DLTensor* dx0, DLTensor* dx1 /*nullable*/, DLTensor* dx2 /*nullable*/,
                               DLTensor* dx3 /*nullable*/, const DLTensor* wpacked, const DLTensor* wpacked_pw,
                               void* stream);
int b3d_conv3d_wgrad_p16(const DLTensor* x0, const DLTensor* x1, const DLTensor* x2, const DLTensor* x3,
                         const DLTensor* dy /*P16*/, DLTensor* dw, int stride, int transposed, DLTensor* scratch,
                         void* stream);
/* both weight gradients of the convs reading a ResnetBlock's input (/root/reference/layers/resnet.py:118 pointwise, :133
 * first 3x3x3) in one pass over x: dw <- (x, dy), dw_pw <- (x, dres).  Only where b3d_conv3d_wgrad_p16_block_ok(cin,
 * cout, H, W) returns 1 (else B3D_ERR_UNSUPPORTED: call b3d_conv3d_wgrad_p16 twice). */
int b3d_conv3d_wgrad_p16_block(const DLTensor* x0, const DLTensor* x1, const DLTensor* x2, const DLTensor* x3,
                               const DLTensor* dy /*P16*/, const DLTensor* dres /*P16*/, DLTensor* dw, DLTensor* dw_pw,
                               void* stream);
int b3d_conv3d_wgrad_p16_block_ok(int cin, int cout, int h_sp, int w_sp);
/* 0: the layer's weight gradient is not on the P16 path; 1: straight from the operands; 2: needs a 16-bit scratch of
 * numel(big tensor) elements (stride-2 family); 3: of numel(dy) elements (TS-mode kernel).  w_sp = W of dy. */
int b3d_conv3d_wgrad_p16_plan(int k, int stride, int transposed, int cin, int cout, int w_sp);

#ifdef __cplusplus
}
#endif
#endif
