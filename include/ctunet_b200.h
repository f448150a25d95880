/*
 * ctunet_b200 -- C ABI of the B200-native (sm_100a) hot path of vfmatzkin/ct-unet.
 *
 * The reference is pure Python/PyTorch and has NO FFI of its own (SURVEY.md section 8b): its hot
 * path is the `torch.nn` module graph built in ctunet/pytorch/models.py plus the loss in
 * ctunet/pytorch/ProblemHandler.py and ctunet/utilities.py.  This header is therefore the
 * boundary a maintainer would bind (ctypes stub in INTEGRATION.md); each entry point cites the
 * reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name starts with `h_` (host array of small
 *    metadata such as a list of source pointers); PyTorch (the caller) owns all memory, the library
 *    never allocates, frees or retains device memory;
 *  - all work is enqueued on `stream` (a cudaStream_t passed as void*); no call synchronises, so
 *    every entry point is CUDA-graph capturable;
 *  - return value: 0 ok, <0 invalid argument / unsupported shape, >0 a cudaError_t; the message
 *    is available (thread-local) from ctu_last_error();
 *  - there is NO CPU fallback.
 *
 * Activation layout ("blocked"): [N][Cb][D][H][W][8], Cb = ceil(C/8); the 8 channels of one
 * voxel are contiguous (16 B in bf16, 32 B in fp32); pad lanes (channel >= C) are always zero.
 * `dtype` selects the storage type of blocked activations: CTU_BF16 is the product mode
 * (fp32 accumulation everywhere), CTU_F32 is the fp32 "accumulate-check" mode of north_star.
 * A convolution / head input may be the channel concatenation of up to CTU_MAX_SRC blocked tensors
 * (the reference's `cat((ubl, d[-i-1]), 1)`, models.py:249, is never materialised): `h_srcs[i]`
 * with `h_src_channels[i]` real channels each, concatenated in order.
 */
#ifndef CTUNET_B200_H
#define CTUNET_B200_H

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define CTU_OK 0
#define CTU_ERR_INVALID (-1)
#define CTU_ERR_UNSUPPORTED (-2)
#define CTU_MAX_SRC 4
/* OR into `use_tensor_path` of ctu_conv3d_fprop / ctu_conv3d_wgrad (there: dwp), `phases` of ctu_bn_stats or `y_phase_major` of
 * ctu_bn_relu_bwd_reduce:
 * the caller has already zeroed the double accumulators (bn_sums / sums / sums2), so the entry point enqueues no memset of
 * its own.  A step driver zeroes ONE arena for all of a pass's accumulators instead of ~30 memset nodes on the layer chain. */
#define CTU_ACCUM_PREZEROED 0x100
#define CTU_DROPOUT_MAX_SITES 32

typedef enum { CTU_F32 = 0, CTU_BF16 = 1 } ctu_dtype;
typedef void* ctu_stream; /* cudaStream_t */

/* head flags (ctu_head_fwd / ctu_head_bwd) */
#define CTU_HEAD_SOFTMAX 1    /* F.softmax(lc, dim=1)            models.py:258, :538 */
#define CTU_HEAD_SIGMOID 2    /* torch.sigmoid(out)              models.py:259       */
#define CTU_HEAD_SP 4         /* UNetSP/UNetDO encode            models.py:319-330   */
#define CTU_HEAD_SP_SOFTMAX 8 /* UNetSPSmall softmax of each pair models.py:364-365  */

const char* ctu_last_error(void);
int ctu_version(void);
/* 1 if the library contains the tcgen05/TMA implicit-GEMM convolution kernels */
int ctu_has_tensor_path(void);

/* ---- layout: fp32 NCDHW (the reference's tensors, Model.py:343) <-> blocked ---------------- */
int ctu_pack_ncdhw(const float* src, void* dst, int dtype, int n, int c, long long spatial, ctu_stream stream);
int ctu_unpack_ncdhw(const void* src, float* dst, int dtype, int n, int c, long long spatial, ctu_stream stream);
/* sliding-window inference (BASELINE config 4): n patches of patch^3 voxels gathered from a float32 [c][vd][vh][vw] volume at
 * the DEVICE int[n][3] origins (z, y, x) into the blocked layout -- no host-side slicing / stacking.  patch % 4 == 0; any
 * volume width and any origin: input voxels outside the volume read as 0 */
int ctu_pack_patches(const float* vol, const int* origins, void* dst, int dtype, int n, int c, int vd, int vh, int vw, int patch,
                     ctu_stream stream);

/* ---- Conv3d k^3, stride 1, "same" zero padding (nn.Conv3d at models.py:26,29,38,41,71,76,
 *      403,407,430,434,483,487), k in {1,3,5}.  Weights are re-packed from the native
 *      [Cout][Cin][k][k][k] fp32 parameter into [cob][cib][tap][ci8][co8] fp32. -------------- */
long long ctu_conv_wpack_floats(int cout, int k, int nsrc, const int* h_src_channels);
int ctu_conv_pack_weight(const float* w, float* wp, int cout, int k, int nsrc, const int* h_src_channels,
                         ctu_stream stream);
/* packed weights of the data-gradient convolution dy -> d(src[which]) (flipped taps, transposed) */
long long ctu_conv_wpack_dgrad_floats(int cout, int k, int src_channels);
int ctu_conv_pack_weight_dgrad(const float* w, float* wpd, int cout, int k, int nsrc, const int* h_src_channels,
                               int which, ctu_stream stream);
int ctu_conv_unpack_wgrad(const float* dwp, float* dw, int cout, int k, int nsrc, const int* h_src_channels,
                          ctu_stream stream);
/* y = conv(cat(srcs)) (+ bias).  The data gradient is the same call on dy with dgrad-packed
 * weights.  bn_sums (nullable, double[2*cpad]): per-channel sum / sum of squares of y for the
 * BatchNorm that follows (fused into the epilogue where possible, so ctu_bn_stats is not needed).
 * stat_cout: 0 (= cout), or the number of NATURAL channels when y is the phase-major output of the
 * fused up-sampling stage (cout = 8 phases x 8*ceil(stat_cout/8); statistics are summed over phases).
 * use_tensor_path: 0 = CUDA-core direct kernel (both dtypes; wp = fp32 packed weights),
 * 1 = tcgen05/TMA implicit GEMM (bf16, shapes accepted by ctu_conv_tc_supported;
 * wp = the bf16 B-tile image written by ctu_conv_tc_pack_weight),
 * 2 = tcgen05/TMA weight-streaming implicit GEMM for wide low-resolution layers (bf16, one source, shapes accepted
 * by ctu_conv_wide_supported; wp = the image written by ctu_conv_wide_pack_weight). */
int ctu_conv3d_fprop(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const void* wp,
                     const float* bias, void* y, double* bn_sums, int stat_cout, int cout, int k, int n, int d, int h,
                     int w, int use_tensor_path, ctu_stream stream);
/* The data gradient (tensor path 1: bf16, wimg from ctu_conv_tc_pack_weight of the dgrad-packed weights) whose output dx is
 * dA of a BatchNorm+ReLU stage that only this convolution consumes (models.py:26-32): the epilogue also reduces the two sums
 * of the BatchNorm backward pass, bn_sums2 = double[2*cpad] = sum(dz) | sum(dz * xhat), dz = dx * [scale*y + shift > 0],
 * from bn_y (the BatchNorm's input, natural layout or phase-major) and bn_ss (as written by ctu_bn_finalize) -- it replaces
 * ctu_bn_relu_bwd_reduce for that stage.  Shapes accepted by ctu_conv_tc_bnred_supported (3x3x3, <= 16 output channels). */
int ctu_conv_tc_bnred_supported(int k, int nsrc, const int* h_src_channels, int cout, int d, int h, int w);
int ctu_conv3d_dgrad_bnred(const void* const* h_srcs, const int* h_src_channels, int nsrc, const void* wimg, void* dx,
                           int cout, int k, int n, int d, int h, int w, const void* bn_y, const float* bn_ss,
                           double* bn_sums2, int bn_y_phase_major, ctu_stream stream);
/* tcgen05 path: coverage predicate, size of the weight image, and the re-pack fp32 packed -> image */
int ctu_conv_tc_supported(int k, int nsrc, const int* h_src_channels, int cout, int d, int h, int w);
int ctu_conv_tc_wgrad_supported(int k, int nsrc, const int* h_src_channels, int cout, int d, int h, int w);
long long ctu_conv_tc_wimg_bytes(int k, int nsrc, const int* h_src_channels, int cout);
int ctu_conv_tc_pack_weight(const float* wp, void* wimg, int k, int nsrc, const int* h_src_channels, int cout,
                            ctu_stream stream);
/* wide tensor path (many channels on a 16^3 / 8^3 grid -- models.py:71,76 center block, :483,487 and the 56..128-channel
 * 5^3 layers of the legacy family): weights streamed tap by tap, h and w multiples of 8.  The image depends on the
 * launch geometry, so the batch and grid sizes are arguments of all three. */
int ctu_conv_wide_supported(int k, int cin, int cout, int n, int d, int h, int w);
long long ctu_conv_wide_wimg_bytes(int k, int cin, int cout, int n, int d, int h, int w);
int ctu_conv_wide_pack_weight(const float* wp, void* wimg, int k, int cin, int cout, int n, int d, int h, int w,
                              ctu_stream stream);
/* weight gradient on 8 x 8 plane tiles (the 8^3 level; h, w multiples of 8, at most 128 input and output channels,
 * one source): ctu_conv3d_wgrad with use_tensor_path = 2 */
int ctu_conv_wide_wgrad_supported(int k, int cin, int cout, int d, int h, int w);
/* dwp (packed layout, fp32) and dbias (nullable, [cout]) are zeroed by the call, then accumulated.
 * phase_cout: 0, or the natural channel count when dy is the phase-major gradient of the fused up-sampling stage
 * COMPOSED FROM A 3x3x3 CONVOLUTION (cout = 8 phases x 8*ceil(phase_cout/8)): the tensor path then skips the taps that are
 * structurally zero (their entries of dwp stay 0 or hold unspecified values that ctu_upfuse_decompose never reads). */
/* use_tensor_path: 0 CUDA cores, 1 conv_tc.cu (16-wide rows, ctu_conv_tc_wgrad_supported), 2 the tap-stationary
 * small-grid kernel (ctu_conv_wide_wgrad_supported). */
int ctu_conv3d_wgrad(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const void* dy,
                     float* dwp, float* dbias, int phase_cout, int cout, int k, int n, int d, int h, int w,
                     int use_tensor_path, ctu_stream stream);

/* ---- ConvTranspose3d k=2, stride 2, with bias (models.py:37, :427).  Native weight
 *      [Cin][Cout][2][2][2]; packed [cob][cib][abc][ci8][co8].  n,d,h,w are the INPUT dims. --- */
long long ctu_convt_wpack_floats(int cout, int nsrc, const int* h_src_channels);
int ctu_convt_pack_weight(const float* w, float* wp, int cout, int nsrc, const int* h_src_channels, ctu_stream stream);
long long ctu_convt_wpack_dgrad_floats(int cout, int src_channels);
int ctu_convt_pack_weight_dgrad(const float* w, float* wpd, int cout, int nsrc, const int* h_src_channels, int which,
                                ctu_stream stream);
int ctu_convt_unpack_wgrad(const float* dwp, float* dw, int cout, int nsrc, const int* h_src_channels,
                           ctu_stream stream);
/* All weight re-packings of a pass in one launch: job j writes dst[i] = idx[i] >= 0 ? src[idx[i]] : 0 for i < counts[j]
 * (dst float32, or bf16 where dst_bf16[j]); counts are multiples of 8; the arrays are HOST arrays of device pointers.  The
 * index maps are the permutations the ctu_conv_*pack_weight* entry points above apply (computed once per layer shape by
 * running them on index-valued inputs), so the result is bit-identical to the chain of packing launches it replaces. */
int ctu_gather_batch(int njobs, const float* const* h_srcs, void* const* h_dsts, const int* const* h_idxs,
                     const long long* h_counts, const int* h_dst_bf16, ctu_stream stream);
int ctu_convt2_fprop(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* wp,
                     const float* bias, void* y, int cout, int n, int d, int h, int w, ctu_stream stream);
int ctu_convt2_dgrad(int dtype, const void* dy, const float* wpd, void* dx, int cout, int src_channels, int n, int d,
                     int h, int w, ctu_stream stream);
int ctu_convt2_wgrad(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const void* dy,
                     float* dwp, float* dbias, int cout, int n, int d, int h, int w, ctu_stream stream);

/* ---- fused up-sampling stage: ConvTranspose3d(k2,s2) followed by Conv3d(k^3,"same") (models.py:37-38, :427-430)
 *      as ONE 3x3x3 convolution on the low-resolution grid with 8 phases x 8*ceil(cout/8) output channels
 *      (output channel q*cop + co, q = qd*4+qh*2+qw); the transposed convolution's bias rides on an extra
 *      all-ones input channel (index cin).  wt [cin][cin][2][2][2], bt [cin] (nullable), w3 [cout][cin][k][k][k],
 *      b3 [cout] (nullable, with b3n [8*cop]);  wn: native [8*cop][cin+1][3][3][3] for ctu_conv_pack_weight. ---- */
int ctu_upfuse_cout(int cout);
/* workspace (caller-owned fp32 scratch of ctu_upfuse_workspace_floats elements): transposed operand copies */
long long ctu_upfuse_workspace_floats(int cin, int cout, int k);
int ctu_upfuse_compose(const float* wt, const float* bt, const float* w3, const float* b3, float* wn, float* b3n, int cin,
                       int cout, int k, float* workspace, ctu_stream stream);
/* chain rule of the composition: dwn [8*cop][cin+1][27] (+ dbn [8*cop]) -> dwt, dbt, dw3 (+ db3) */
int ctu_upfuse_decompose(const float* dwn, const float* dbn, const float* wt, const float* bt, const float* w3, float* dwt,
                         float* dbt, float* dw3, float* db3, int cin, int cout, int k, float* workspace, ctu_stream stream);

/* ---- BatchNorm3d (+ReLU, + MaxPool3d(2,2)) (models.py:27-28,31-32,39-40,43-44,190-191,233) ---
 * sums: double[2*cpad] = per-channel sum and sum of squares (zeroed by ctu_bn_stats).
 * ss:   float[4*cpad]  = scale | shift | mean | invstd, cpad = 8*ceil(c/8).                    */
/* phases: 1, or 8 when y is phase-major (8 copies of the ceil(c/8) natural channel blocks) */
int ctu_bn_stats(int dtype, const void* y, int c, int phases, int n, long long spatial, double* sums, ctu_stream stream);
int ctu_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float* running_mean,
                    float* running_var, long long* num_batches_tracked, float momentum, float eps, int c,
                    int training, int n_updates, float* ss, ctu_stream stream);
/* extra running-stat update(s) with the same batch statistics: the reentrant-checkpoint
 * recomputation of models.py:232 (SURVEY.md Appendix D.2) */
int ctu_bn_running_update(const double* sums, double count, float* running_mean, float* running_var,
                          long long* num_batches_tracked, float momentum, int c, int n_updates, ctu_stream stream);
/* a = relu(scale*y+shift); if pooled != NULL also pooled = maxpool2(a) (d,h,w even).
 * y_phase_major: y (and dy in the backward calls) is [n][8*cb][d/2][h/2][w/2][8], the output layout of the fused
 * up-sampling stage; a / dA stay natural [n][cb][d][h][w][8]; d,h,w are always the natural (high-res) dims. */
int ctu_bn_relu_fwd(int dtype, const void* y, const float* ss, void* a, void* pooled, int c, int n, int d, int h, int w,
                    int y_phase_major, ctu_stream stream);
/* training mode, ctu_bn_finalize folded in: scale / shift come from the batch sums inside the kernel, which also writes
 * ss [4*cpad] for the backward pass and moves running_mean / running_var / num_batches_tracked (nullable) n_updates times */
int ctu_bn_relu_fwd_train(int dtype, const void* y, const double* sums, double count, const float* gamma, const float* beta,
                          float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                          int n_updates, float* ss, void* a, void* pooled, int c, int n, int d, int h, int w,
                          int y_phase_major, ctu_stream stream);
/* _drop variants: keep (nullable, float[n][cpad]) = the Dropout3d keep factors k[n][c] of the site that follows the ReLU
 * (ctu_dropout3d_keep): a = round(k * relu(scale*y + shift)) and pooled = maxpool2 of those values.  The backward variants
 * take the same factors: dz = k * (dA + unpool(dP)) * [scale*y + shift > 0].  NULL = the plain entry points above / below.
 * A phase-major y never precedes a dropout site and is refused with keep != NULL. */
int ctu_bn_relu_fwd_drop(int dtype, const void* y, const float* ss, void* a, void* pooled, int c, int n, int d, int h,
                         int w, int y_phase_major, const float* keep, ctu_stream stream);
int ctu_bn_relu_fwd_train_drop(int dtype, const void* y, const double* sums, double count, const float* gamma,
                               const float* beta, float* running_mean, float* running_var, long long* num_batches_tracked,
                               float momentum, float eps, int n_updates, float* ss, void* a, void* pooled, int c, int n,
                               int d, int h, int w, int y_phase_major, const float* keep, ctu_stream stream);
int ctu_bn_relu_bwd_reduce_drop(int dtype, const void* y, const float* ss, const void* dA, const void* dP, double* sums2,
                                int c, int n, int d, int h, int w, int y_phase_major, const float* keep, ctu_stream stream);
int ctu_bn_relu_bwd_apply_drop(int dtype, const void* y, const float* ss, const float* gamma, const void* dA, const void* dP,
                               const double* sums2, double count, void* dy, float* dgamma, float* dbeta, int c, int n, int d,
                               int h, int w, int y_phase_major, const float* keep, ctu_stream stream);
/* Dropout3d keep factors of the nsite sites of one pass (nsite <= CTU_DROPOUT_MAX_SITES), site i at
 * keep + n * (cpad_0 + ... + cpad_{i-1}) as float[n][cpad_i], cpad_i = 8*ceil(h_channels[i]/8):
 * k = 1/(1-p) with probability 1-p, else 0 (p = 1: all zero; pad lanes 0).  Philox4x32-10 keyed by `seed`, counter =
 * (pass, h_site[i], sample*cpad_i + channel) with pass = *pass_counter, which the launch then advances by one (so a replayed
 * CUDA graph draws new masks every replay); pass_counter NULL: pass 0, nothing advanced.  One block, no host sync. */
int ctu_dropout3d_keep(int nsite, const int* h_site, const int* h_channels, const float* h_p, int n,
                       unsigned long long seed, unsigned long long* pass_counter, float* keep, ctu_stream stream);
/* backward, pass 1: sums2 = double[2*cpad] = sum(dz), sum(dz*xhat) with
 * dz = (dA + unpool(dP)) * [a > 0]; dA and dP are nullable (not both) */
int ctu_bn_relu_bwd_reduce(int dtype, const void* y, const float* ss, const void* dA, const void* dP, double* sums2,
                           int c, int n, int d, int h, int w, int y_phase_major, ctu_stream stream);
/* backward, pass 2: dy, dgamma[c], dbeta[c] */
int ctu_bn_relu_bwd_apply(int dtype, const void* y, const float* ss, const float* gamma, const void* dA, const void* dP,
                          const double* sums2, double count, void* dy, float* dgamma, float* dbeta, int c, int n, int d,
                          int h, int w, int y_phase_major, ctu_stream stream);

/* ---- head: last_conv 1x1x1 + bias (models.py:224,255 / :507,535), optional softmax / sigmoid,
 *      UNetSP encode.  w is the NATIVE [cout][cin_total] fp32 parameter.  Outputs are fp32 NCDHW:
 *      out0 = [n][cout] planes (plain) or the encoded full skull [n][2]; out1 = encoded flap. --- */
int ctu_head_fwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                 const float* bias, int cout, int flags, float* out0, float* out1, int n, long long spatial,
                 ctu_stream stream);
/* head + hard_segm_from_tensor (utilities.py:103-124) in one kernel: float32 labels = argmax over the channels of every head
 * output (first maximum wins, as ctu_argmax_channels).  origins == NULL: labels0 / labels1 are [n][spatial] planes;
 * origins = DEVICE int[n][3]: every sample is a patch^3 patch scattered into the [vd][vh][vw] label volumes at its origin
 * (the stitch of a sliding-window pass).  labels1 only for the SP heads. */
int ctu_head_labels(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w, const float* bias,
                    int cout, int flags, const int* origins, int patch, int vd, int vh, int vw, float* labels0, float* labels1,
                    int n, long long spatial, ctu_stream stream);
/* Overlapping sliding-window inference (DESIGN.md section 7b): the head of every patch^3 window at the DEVICE origins adds
 * llrint(w * v * 2^40) to the int64 accumulators acc[out][c][vd][vh][vw] for each output channel value v (what
 * ctu_head_fwd writes) of every window voxel inside the volume, with w = weights[z] * weights[patch + y] *
 * weights[2*patch + x] (DEVICE float[3][patch]).  Integer atomics: the sums are independent of the order of the windows.
 * The head must be bounded (softmax or sigmoid): every v lies in [0, 2]. */
int ctu_head_accumulate(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                        const float* bias, int cout, int flags, const int* origins, int patch, int vd, int vh, int vw,
                        const float* weights, long long* acc, int n, long long spatial, ctu_stream stream);
/* labels[o] = float32 argmax over the channels of acc[o] (first maximum wins) for n_out = 1 or 2 outputs of `channels`
 * channels each; probs[o] (nullable) = float32 [channels][vd][vh][vw] acc * 2^-40 / (nz[z] * ny[y] * nx[x]) with the
 * DEVICE float64 normaliser tables norm = [nz (vd) | ny (vh) | nx (vw)]. */
int ctu_window_finalize(const long long* acc, int n_out, int channels, int vd, int vh, int vw, const double* norm,
                        float* labels0, float* labels1, float* probs0, float* probs1, ctu_stream stream);
/* dsrcs[i] nullable; dw [cout][cin_total] and db [cout] are zeroed by the call.  dw = db = NULL: source gradients only;
 * every dsrcs[i] NULL: parameter gradients only (two launches that can run on different streams) */
/* out0 / out1 (nullable): the outputs ctu_head_fwd produced; with them the plain-sigmoid SP head skips the logits */
int ctu_head_bwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                 const float* bias, int cout, int flags, const float* dout0, const float* dout1, const float* out0,
                 const float* out1, void* const* h_dsrcs,
                 float* dw, float* db, int n, long long spatial, ctu_stream stream);

/* ---- fused head + loss for the training step (models.py:255-259, 319-330, 535-538 + ProblemHandler.py:59-91, 228-298):
 *      the head is recomputed from the blocked sources and fed to the Dice + CrossEntropy arithmetic in registers, so the
 *      fp32 network outputs and their gradients never touch HBM.  target0 / target1: one-hot float32 [n][C][spatial]
 *      (SP heads: two targets with C = 2; plain head: target0 with C = cout, target1 = NULL); with target_u8 the targets
 *      are uint8 class-1 masks [n][spatial] instead (two classes: the label volumes of datasets.py:209-214 before the
 *      one-hot encoding -- 1 byte per voxel and target instead of 8).  softmax_for_dice as
 *      ctu_dice_ce_fwd.  sums: double[4 * pairs * n] (zeroed by the forward call, read by the backward calls).
 *      comps: float[terms + 1] = [ce_lambda * CE per pair] (if ce_lambda != 0) + [dice_lambda * Dice per pair]
 *      (if dice_lambda != 0) + [total]; mirror (nullable): a second copy (tail of the data-parallel gradient buffer). */
int ctu_head_loss_fwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                      const float* bias, int cout, int flags, const void* target0, const void* target1, int target_u8,
                      int softmax_for_dice, float ce_lambda, float dice_lambda, double* sums, float* comps, float* mirror,
                      int n, long long spatial, ctu_stream stream);
/* d(total) / d(sources) into h_dsrcs; also stores the logit gradients dlogits [n][cout][spatial] (fp32) for
 * ctu_head_param_grad, which reduces dW [cout][cin_total] and db [cout] (zeroed by the call) from them and the sources --
 * a leaf of the backward pass that can run on another stream. */
int ctu_head_loss_bwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                      const float* bias, int cout, int flags, const void* target0, const void* target1, int target_u8,
                      int softmax_for_dice, float ce_lambda, float dice_lambda, const double* sums, void* const* h_dsrcs,
                      float* dlogits, int n, long long spatial, ctu_stream stream);
int ctu_head_param_grad(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* dlogits,
                        int cout, float* dw, float* db, int n, long long spatial, ctu_stream stream);

/* ---- loss: soft Dice (utilities.py:39-50) + CrossEntropy (ProblemHandler.py:67-70, 247-257) on
 *      one prediction/target pair, fp32 NCDHW [b][c][spatial], c <= 4.
 * sums: double[4*b] (zeroed by the call): sum p*t, sum p*p, sum t*t, CE sum.
 * out:  float[2] = { ce_mean, dice_loss }.                                                      */
int ctu_dice_ce_fwd(const float* pred, const float* target, int b, int c, long long spatial, int softmax_for_dice,
                    int want_ce, double* sums, float* out, ctu_stream stream);
/* dpred = g[0] * dCE/dpred + g[1] * dDice/dpred; g is a DEVICE float[2] */
int ctu_dice_ce_bwd(const float* pred, const float* target, int b, int c, long long spatial, int softmax_for_dice,
                    int want_ce, const double* sums, const float* g, float* dpred, ctu_stream stream);

/* ---- hard segmentation: argmax over channels as float32, ties -> lowest index
 *      (utilities.py:103-124) ------------------------------------------------------------------ */
int ctu_argmax_channels(const float* x, float* out, int b, int c, long long spatial, ctu_stream stream);

/* ---- virtual craniectomy (transforms.py:241-300, utilities.py:127-178), uint8 volumes -------- */
/* count[0] = number of voxels > 0 (np.argwhere(image > 0).shape[0], transforms.py:249) */
int ctu_count_nonzero_u8(const unsigned char* img, long long nvox, long long* count, ctu_stream stream);
/* coords[0..2] = np.argwhere(img > 0)[k] in C order; block_counts is scratch: long long[ceil(nvox/4096)+1] */
int ctu_kth_nonzero_u8(const unsigned char* img, int d, int h, int w, long long k, long long* block_counts, int* coords,
                       ctu_stream stream);
/* shape: 0 sphere (2-norm), 1 box (inf-norm), 2 flap (two cylinders of radius c_diam + a cube, utilities.py:145-166;
 * restates raster_geometry.cylinder / cube, which the reference imports un-vendored: parity unpinned);
 * centre read from DEVICE int[3]; masked = img AND outside, extracted = img AND inside (distance <= size, float64
 * like numpy).  c_diam is only read for shape 2. */
int ctu_flap_mask_u8(const unsigned char* img, unsigned char* masked, unsigned char* extracted, int d, int h, int w,
                     const int* center, double size, int shape, double c_diam, ctu_stream stream);

/* (skull_target = flap_target = NULL: the image only -- the fused head + loss kernels read the uint8 label masks directly) */
/* ---- batch encoding on the device (datasets.py:195-235, :30-47): uint8 masks [batch][spatial] ->
 *      image [batch][in_channels][spatial] float32 (channel 0 = broken skull, channel 1 = atlas [spatial], nullable for
 *      1-channel models) and the two one-hot float32 targets [batch][2][spatial] (datasets.py:209-214). ---------- */
int ctu_encode_flaprec_u8(const unsigned char* broken, const unsigned char* full, const unsigned char* flap,
                          const float* atlas, float* image, float* skull_target, float* flap_target, int batch,
                          int in_channels, long long spatial, ctu_stream stream);

/* the same from BIT-PACKED masks [batch][spatial / 8] (voxel v = bit v & 7 of byte v >> 3: numpy packbits, bitorder
 * "little"): image as above, and (nullable, both or neither) the uint8 label masks [batch][spatial] that
 * ctu_head_loss_fwd / _bwd take with target_u8 = 1.  Binary volumes cross PCIe at 3 bits per voxel. */
int ctu_encode_flaprec_bits(const unsigned char* broken_bits, const unsigned char* full_bits, const unsigned char* flap_bits,
                            const float* atlas, float* image, unsigned char* full_mask, unsigned char* flap_mask, int batch,
                            int in_channels, long long spatial, ctu_stream stream);

/* ---- CT preprocessing (no reference implementation: oracle/unet_oracle.py defines it) -------- */
int ctu_hu_window(const short* hu, float* out, long long nvox, float lo, float hi, ctu_stream stream);
int ctu_hu_threshold(const short* hu, unsigned char* out, long long nvox, int thr, ctu_stream stream);
int ctu_resample_nearest_f32(const float* src, float* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                             ctu_stream stream);
int ctu_resample_nearest_u8(const unsigned char* src, unsigned char* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                            ctu_stream stream);
int ctu_resample_nearest_index(int* idx, int out_size, int in_size, ctu_stream stream);
int ctu_resample_trilinear_f32(const float* src, float* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                               ctu_stream stream);

/* ---- connected components of [b][d][h][w] volumes (scipy.ndimage.label semantics; DESIGN.md section 7c).  A voxel is
 *      foreground when it is non-zero; in_dtype is CTU_MASK_U8 (uint8 or bool) or CTU_MASK_F32 (float32, e.g. the label
 *      volumes of the sliding-window functions).  connectivity 6, 18 or 26 = generate_binary_structure(3, 1 / 2 / 3);
 *      b*d*h*w < 2^31.  Each volume is labelled on its own.  ws: caller-owned DEVICE scratch of
 *      ctu_components_workspace_bytes(b, d, h, w) bytes, 16-byte aligned (-1: invalid shape). */
#define CTU_MASK_U8 1
#define CTU_MASK_F32 4
long long ctu_components_workspace_bytes(int b, int d, int h, int w);
/* labels int32 [b][d][h][w]: 0 background, components 1..n per volume in the raster order of their first voxel;
 * counts int64 [b] = n per volume. */
int ctu_label_components(int in_dtype, const void* in, int b, int d, int h, int w, int connectivity, int* labels,
                         long long* counts, void* ws, long long ws_bytes, ctu_stream stream);
/* out (same dtype and shape as in) = in, except 0 on the voxels of dropped components.  min_size >= 0: keep every
 * component of at least min_size voxels; min_size < 0: keep only the largest component of each volume (ties: the one
 * whose first voxel comes first in raster order). */
int ctu_filter_components(int in_dtype, const void* in, int b, int d, int h, int w, int connectivity, long long min_size,
                          void* out, void* ws, long long ws_bytes, ctu_stream stream);

/* ---- reporting metrics of the loss handlers (utilities.py:53-70; ProblemHandler.py:84-88, 277-295) on fp32 NCDHW
 *      prediction / one-hot target pairs [b][c][spatial], 2 <= c <= 4.  monai (undeclared, unpinned in the reference) is
 *      restated: PARITY UNPINNED, the CPU statement is oracle/ref_stubs/monai/metrics.py. -------------------------------- */
/* out[0] = torch.mean(compute_meandice(one_hot(argmax(pred,1)), target, include_background=False)):
 * per (sample, class >= 1) 2*sum(t*m)/(sum(t)+sum(m)), NaN where sum(t) == 0.  counts: double[3*b*(c-1)] scratch. */
int ctu_dice_coeff(const float* pred, const float* target, int b, int c, long long spatial, double* counts, float* out,
                   ctu_stream stream);
/* out[0] = mean over (sample, class >= 1) of the symmetric Hausdorff distance between the surfaces (mask minus its
 * 6-neighbourhood erosion) of [argmax(pred) == class] and [target[class] == 1]; exact squared Euclidean distance
 * transform in int32; an empty surface on either side counts as inf_alt (= max(target.shape), utilities.py:64,69). */
long long ctu_hausdorff_workspace_bytes(int b, int c, int d, int h, int w);
int ctu_hausdorff(const float* pred, const float* target, int b, int c, int d, int h, int w, double inf_alt, void* workspace,
                  long long workspace_bytes, double* out, ctu_stream stream);

/* ---- surface-distance evaluation of binary masks (DESIGN.md section 7d).  pred and target: [b][d][h][w], each
 *      CTU_MASK_U8 (uint8 or bool) or CTU_MASK_F32, non-zero = foreground; every axis 1..1024, b*d*h*w < 2^31.  Edges are
 *      the mask minus its 6-neighbourhood erosion (outside = background); d(A->B) = the Euclidean distances from the edge
 *      voxels of A to the nearest edge voxel of B, in voxel units (spacing NULL) or weighted by spacing = host double[3]
 *      (sz, sy, sx), positive and finite.  out: DEVICE double[5][b], rows dice (2|P n T| / (|P| + |T|)), hausdorff (max of
 *      both directed maxima), hausdorff_percentile (max over both directions of numpy.percentile(d, percentile), method
 *      "linear"), assd (mean of both directed distance sets together), surface_dice (#{d <= tolerance} over both
 *      directions / (#edges(P) + #edges(T))).  Both masks empty: all NaN; one empty: dice and surface_dice 0, distances
 *      +inf.  0 <= percentile <= 100, tolerance >= 0.  No host synchronisation; the same inputs give the same bits.
 *      ws: DEVICE scratch of ctu_surface_metrics_workspace_bytes(b, d, h, w, spacing != NULL) bytes, 8-byte aligned
 *      (-1: invalid shape). */
long long ctu_surface_metrics_workspace_bytes(int b, int d, int h, int w, int weighted);
int ctu_surface_metrics(int pred_dtype, const void* pred, int target_dtype, const void* target, int b, int d, int h, int w,
                        const double* spacing, double percentile, double tolerance, double* out, void* ws, long long ws_bytes,
                        ctu_stream stream);

/* ---- the tail of a training iteration (Model.py:366-371, 510-546; ProblemHandler.py:59-91, 241-298) -------------------
 * comps[i] = lambdas[i] * *terms[i] (device scalars, host array of pointers), comps[n] = their sum in order; mirror
 * (nullable) receives a second copy (the tail of the data-parallel flat gradient buffer). */
int ctu_loss_combine(const float* const* h_terms, const float* h_lambdas, int n, float* comps, float* mirror,
                     ctu_stream stream);
/* One launch updates every parameter.  chunks: device array of n_chunks records {float* param; long long flat_off; int count;
 * int pad;} (ctu_optim_chunk_bytes() each, count <= ctu_optim_chunk_elems()) mapping pieces of the parameter tensors to
 * offsets of the flat gradient / state buffers.  kind: 0 Adam, 1 AdamW (state0 exp_avg, state1 exp_avg_sq, state2
 * max_exp_avg_sq when amsgrad), 2 RMSprop (state0 square_avg, state1 momentum buffer), 3 SGD (state0 momentum buffer).
 * lr (device double) and step (device counter of completed steps) are read, not written: ctu_optim_post advances the
 * counter and, with use_plateau, applies torch's ReduceLROnPlateau.step(loss) to sched_state = double[10]
 * { lr, best, num_bad_epochs, cooldown_counter, factor, patience, threshold, min_lr, cooldown, eps } -- lr = sched_state. */
int ctu_optim_chunk_bytes(void);
int ctu_optim_chunk_elems(void);
int ctu_optim_step(int kind, const void* chunks, int n_chunks, const float* flat_grad, float* state0, float* state1,
                   float* state2, const double* lr, const long long* step, double beta1, double beta2, double eps,
                   double weight_decay, double momentum, double alpha, int amsgrad, double grad_scale, ctu_stream stream);
int ctu_optim_post(long long* step, double* sched_state, const float* loss, int use_plateau, ctu_stream stream);

/* ---- data-parallel gradient exchange fused with the optimizer over NVLink peer memory (replaces nn.DataParallel's
 *      reduce / broadcast, Model.py:481-486; one process per GPU).  Every rank's flat gradient buffer lives in an
 *      IPC-shared allocation: [flag page of ctu_peer_flag_bytes()] [flat fp32 gradients | loss tail].  h_grads[r] / h_flags[r]:
 *      HOST arrays of the world's device pointers as mapped into THIS process (own rank included). ---------------------- */
int ctu_peer_flag_bytes(void);
/* setup-time only (the step itself never allocates): cudaMalloc + zero + cudaIpcGetMemHandle / OpenMemHandle */
int ctu_peer_alloc(long long bytes, void** ptr, unsigned char* handle64);
int ctu_peer_open(const unsigned char* handle64, void** ptr);
int ctu_peer_close(void* ptr);
int ctu_peer_free(void* ptr);
/* after the last gradient kernel of a step: publish "my gradients of step seq+1 are complete" to every peer */
int ctu_peer_signal(const void* const* h_grads, void* const* h_flags, int world, int rank, ctu_stream stream);
/* before the first gradient write of a step: every peer has finished reading this rank's previous gradients */
int ctu_peer_wait_done(const void* const* h_grads, void* const* h_flags, int world, int rank, ctu_stream stream);
/* ctu_optim_step with the gradient of element f = mean over ranks (summed in rank order) of h_grads[r][f], read through
 * the peer pointers once every rank has signalled; also averages the tail_n loss floats at tail_off into tail_out and
 * releases the peers' buffers.  One launch = all-reduce + optimizer. */
int ctu_optim_step_peer(int kind, const void* chunks, int n_chunks, const void* const* h_grads, void* const* h_flags, int world,
                        int rank, float* state0, float* state1, float* state2, const double* lr, const long long* step,
                        double beta1, double beta2, double eps, double weight_decay, double momentum, double alpha, int amsgrad,
                        double grad_scale, float* tail_out, long long tail_off, int tail_n, ctu_stream stream);
/* host read (synchronises): 0 ok, 1 a peer's gradients never arrived, 2 a peer never released this rank's buffer */
int ctu_peer_error(const void* flags);

/* ---- SaltAndPepper (transforms.py:13-49) on a uint8 volume: out = (img AND black) OR white with
 *      black = (u_b > density*(1-salt_ratio)), white = 1 - (u_w > density*salt_ratio).  u_black / u_white: caller-supplied
 *      float64 uniform fields (both or neither); NULL = Philox4x32-10 keyed by seed, counter = offset + voxel index. ------ */
int ctu_salt_pepper_u8(const unsigned char* img, unsigned char* out, long long nvox, double noise_density, double salt_ratio,
                       const double* u_black, const double* u_white, unsigned long long seed, unsigned long long offset,
                       ctu_stream stream);

/* ---- random affine augmentation of mask batches (no reference counterpart: the reference has no spatial augmentation;
 *      DESIGN.md section 7e).  Volumes [batch][d][h][w], 1 <= batch <= 65535, every axis below 2^22.
 *      A sample's map from output voxel p = (z, y, x) to source point is q = c + t + (1/s) R F (p - c), c = (S - 1) / 2,
 *      R = R_d(a_d) R_h(a_h) R_w(a_w) (R_a: rotation about axis a), F = diag(f_z, f_y, f_x), f = +-1; matrices = DEVICE
 *      float[batch][3][4] rows (M_k0, M_k1, M_k2, M_k3).  Nearest neighbour in float32 without contraction:
 *      q_k = ((M_k0 z + M_k1 y) + M_k2 x) + M_k3, i_k = floor(q_k + 0.5); the voxel reads 0 unless -0.5 < q_k < S_k - 0.5
 *      on every axis (NaN / inf fail the test).  Every mask of a sample uses the same source index. ------------------ */
/* params = DEVICE float[batch][10] (a_d, a_h, a_w in radians, s, t_z, t_y, t_x, f_z, f_y, f_x) and the matrices they give
 * (built in double, rounded once).  h_ranges = HOST float[8]: max |angle| about d, h, w in [0, pi] (radians), scale lo,
 * hi (0 < lo <= hi), max |translation| along z, y, x (voxels); angle = r (2u - 1), s = lo + (hi - lo) u, t = T (2u - 1),
 * axis k flips when bit k of flip_axes is set and u < 0.5, u = 24-bit uniforms of Philox4x32-10 with counter = (pass,
 * sample, call 0..2) and key = seed.  pass_counter: DEVICE int64 read, then advanced by the launch (NULL: pass 0). */
int ctu_affine_draw(int batch, int d, int h, int w, const float* h_ranges, int flip_axes, unsigned long long seed,
                    unsigned long long* pass_counter, float* params, float* matrices, ctu_stream stream);
/* ctu_encode_flaprec_u8 (bits = 0: uint8 masks [batch][spatial]) / ctu_encode_flaprec_bits (bits = 1: bit-packed
 * [batch * spatial / 8]) with the masks transformed: image channel 0 = transformed broken mask as float, channel 1 = the
 * atlas UNCHANGED (the fixed shape prior in atlas space), full_mask / flap_mask = the transformed uint8 label masks. */
int ctu_affine_encode_flaprec(int bits, const unsigned char* broken, const unsigned char* full, const unsigned char* flap,
                              const float* atlas, const float* matrices, float* image, unsigned char* full_mask,
                              unsigned char* flap_mask, int batch, int in_channels, int d, int h, int w, ctu_stream stream);
/* the same gather for n = 1..3 uint8 masks: h_dst[i] = transformed h_src[i] (HOST arrays of device pointers) */
int ctu_affine_masks_u8(int n, const unsigned char* const* h_src, unsigned char* const* h_dst, const float* matrices,
                        int batch, int d, int h, int w, ctu_stream stream);

/* ---- virtual craniectomy drawn on the device (DESIGN.md section 7f): per sample the distribution of
 *      random_blank_patch(full, p, True, p_type="random", valid_shapes) (transforms.py:241-300) from a Philox stream
 *      instead of the host RNGs.  full = the full-skull masks, uint8 [batch][d][h][w] (bits = 0; non-zero is bone) or
 *      bit-packed [batch * d*h*w / 8] (bits = 1, as ctu_encode_flaprec_bits); 1 <= batch <= 65535, every axis 1..16384.
 *      params = DEVICE double[batch][7] (applied, shape, radius, c_diam, z, y, x): shape 0 sphere / 1 box / 2 flap as
 *      ctu_flap_mask_u8, the integer radius, c_diam for the flap (0 otherwise), the centre voxel (-1s when not applied).
 *      params is 8-byte aligned; `full` has no alignment requirement (a bit-packed view may start at any byte).
 *      Philox4x32-10 with key = seed and counter = (pass, sample, call); the words r[call][0..3] feed:
 *        call 0: gate u = u53(r0, r1) (applied iff u <= p and the skull has bone), k = floor((r2 | r3 << 32) * n / 2^64)
 *                -> centre = np.argwhere(full > 0)[k] (n bone voxels, C order)
 *        call 1: radius = min_radius + floor((r0 | r1 << 32) * (max_radius - min_radius) / 2^64); shape = the enabled
 *                shape (bit 0 sphere, 1 box, 2 flap of `shapes`) of rank floor((r2 | r3 << 32) * popcount(shapes) / 2^64)
 *        call 2: c_diam = ((0.25 + 0.75 u53(r0, r1)) * radius) / 4 (flap only)
 *      with u53(a, b) = ((a >> 5) 2^26 + (b >> 6)) / 2^53.  ws: DEVICE scratch of ctu_craniectomy_workspace_bytes bytes,
 *      16-byte aligned (-1: invalid shape).  Two launches (per-chunk bone counts, then one CTA for the batch);
 *      pass_counter: DEVICE int64 read, then advanced (NULL: pass 0).  min_radius < max_radius, 0 <= p <= 1. */
long long ctu_craniectomy_workspace_bytes(int batch, int d, int h, int w);
int ctu_craniectomy_draw(int bits, const unsigned char* full, int batch, int d, int h, int w, double p, int shapes,
                         int min_radius, int max_radius, unsigned long long seed, unsigned long long* pass_counter,
                         double* params, void* ws, long long ws_bytes, ctu_stream stream);
/* ctu_affine_encode_flaprec from the full skull alone, the hole cut in source space: for output voxel p with source voxel s
 * (matrices as ctu_affine_encode_flaprec, or NULL: s = p), full = (full[s] != 0), inside = the hole of params (as
 * ctu_craniectomy_draw writes them) at s with the arithmetic of ctu_flap_mask_u8; image channel 0 = full AND NOT inside as
 * float, channel 1 = the atlas unchanged, full_mask = full, flap_mask = full AND inside (uint8). */
int ctu_craniectomy_encode_flaprec(int bits, const unsigned char* full, const double* params, const float* atlas,
                                   const float* matrices, float* image, unsigned char* full_mask, unsigned char* flap_mask,
                                   int batch, int in_channels, int d, int h, int w, ctu_stream stream);
/* the same cut as uint8 masks, no transform: broken = full AND NOT inside, full_out = full, flap = full AND inside */
int ctu_craniectomy_masks_u8(const unsigned char* full, const double* params, unsigned char* broken, unsigned char* full_out,
                             unsigned char* flap, int batch, int d, int h, int w, ctu_stream stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CTUNET_B200_H */
