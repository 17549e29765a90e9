/* ptta_b200.h -- C ABI of the B200-native ProxyTTA adaptation step (libptta_b200.so).
 *
 * Drop-in boundary for seobbro/TTA-depth-completion's per-frame TTA step.  The reference has no C
 * FFI of its own for MSG-CHN (it is PyTorch eager: src/external_model_adapt.py:82-237,371-441,
 * src/msg_chn_model_adapt.py:32-125, external_src/MSG_CHN/workspace/exp_msg_chn/
 * network_exp_msg_chn_adapt.py:337-557) and one pybind11 module for NLSPN's deformable conv
 * (external_src/NLSPN/src/model/deformconv/src/vision.cpp:6-13).  Every entry point below names the
 * reference code it replaces.  Conventions:
 *   - plain C: raw DEVICE pointers, ints, floats, a cudaStream_t passed as void*; no torch types;
 *   - every function returns 0 on success; on failure a message is available from ptta_last_error();
 *   - nothing allocates device memory behind the caller's back: the engine reports the workspace it
 *     needs (ptta_msgchn_workspace_bytes) and the caller binds a buffer of that size;
 *   - all work is enqueued on the given stream; nothing synchronises unless stated;
 *   - 32-channel feature maps are NHWC bf16, single-channel maps fp32 [N,H,W], images fp32 NCHW.
 */
#ifndef PTTA_B200_H
#define PTTA_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* ptta_stream_t;            /* cudaStream_t */
typedef struct ptta_msgchn ptta_msgchn; /* opaque engine */
typedef struct ptta_comm ptta_comm;     /* peer communicator of the shared-model mode (below) */

const char* ptta_last_error(void);
int ptta_version(void);

/* ---- stand-alone operators (also the units the parity tests exercise) ------------------------- */

/* src/tta_main.py:583-586 (validity map) + src/net_utils.py:766-811 (OutlierRemoval.remove_outliers) */
int ptta_outlier_removal(const float* sparse_depth, float* filtered_depth, float* filtered_validity,
                         int n, int h, int w, int kernel_size, float threshold, ptta_stream_t stream);
/* src/external_model_adapt.py:103-108 (clamp) + network_exp_msg_chn_adapt.py:479,487,492 (pyramid) */
int ptta_pyramid(const float* depth, float* depth_clamped, float* depth_half, float* depth_quarter,
                 int n, int h, int w, float max_input_depth, int do_clamp, ptta_stream_t stream);
/* fp32 conv weight -> bf16 [tap][O][I] operand; strides in elements, flip reverses the 3x3 taps */
int ptta_pack_conv_weight(const float* src, void* dst_bf16, int o, int i, int stride_o, int stride_i, int flip,
                          ptta_stream_t stream);
/* F.conv2d / F.conv_transpose2d 3x3 (network_exp_msg_chn_adapt.py:166-311) and their data gradients.
 * mode: 0 stride 1, 1 stride 2, 2 transposed stride 2.  prologue: 0 none, 1 ReLU, 2 BN-affine+LeakyReLU.
 * mask_mode: 0 none, 1 [mask>0], 2 LeakyReLU'(mask*mask_scale+mask_shift).  out = add + mask*(conv+bias). */
int ptta_conv3x3(const void* in_bf16, void* out_bf16, const void* wpack_bf16, const float* bias,
                 int n, int hin, int win, int cin, int cout, int mode,
                 int prologue, const float* pro_scale, const float* pro_shift, float slope,
                 const void* mask_bf16, int mask_mode, const float* mask_scale, const float* mask_shift,
                 const void* add_bf16, ptta_stream_t stream);
/* the 32->32 stride-1 case of ptta_conv3x3 on the tcgen05 tensor cores (TMA-fed SWIZZLE_128B pixel-pair rows, TMEM
 * accumulators).  wimage = ptta_pack_conv_weight_tc(wpack): the 18 KB shared-memory image of the [9][32][32] pack.
 * W must be even; relu_in must be 0 (producers store ReLU(x) via relu_out); mask semantics: out = add + [mask>0]*(conv+bias) */
int ptta_pack_conv_weight_tc(const void* wpack_bf16, void* wimage_bf16, ptta_stream_t stream);
int ptta_conv3x3_tc(const void* in_bf16, void* out_bf16, const void* wimage_bf16, const float* bias, int n, int h, int w,
                    int relu_in, int relu_out, const void* mask_bf16, const void* add_bf16, ptta_stream_t stream);
/* same with the two fused extras the engine uses: out2 (optional) = ReLU(bf16(out) [+ add2]) -- the ReLU'd copy a following tensor-core
 * conv reads, or the decoder sum s = ReLU(conv + skip) (network_exp_msg_chn_adapt.py:301-309).  add and add2 are mutually exclusive. */
int ptta_conv3x3_tc_ex(const void* in_bf16, void* out_bf16, void* out2_bf16, const void* wimage_bf16, const float* bias, int n, int h, int w,
                       int relu_out, const void* mask_bf16, const void* add_bf16, const void* add2_bf16, ptta_stream_t stream);
/* out = conv(in) + bias + up2(half) with up2 = F.interpolate(scale_factor=2, bilinear, align_corners=True) of the half-resolution map
 * half [n, h/2, w/2, 32] (the cascade's `x = conv(.) + up(pre_x)`, network_exp_msg_chn_adapt.py:172-186, in ONE pass); out_relu (optional) = ReLU(out) */
int ptta_conv3x3_tc_up2(const void* in_bf16, void* out_bf16, void* out_relu_bf16, const void* weight_image, const float* bias,
                        const void* half_bf16, int n, int h, int w, ptta_stream_t stream);
/* the 32->32 STRIDE-2 case (mode 1 of ptta_conv3x3: Conv2d(s2) forward, ConvTranspose2d(s2) data gradient) on tcgen05.
 * h, w = input size (even); out is [n, h/2, w/2, 32]; out_relu (optional) additionally receives ReLU(out). */
int ptta_pack_conv_weight_tc_s2(const void* wpack_bf16, void* wimage_bf16, ptta_stream_t stream);
int ptta_conv3x3_tc_s2(const void* in_bf16, void* out_bf16, void* out_relu_bf16, const void* wimage_bf16, const float* bias,
                       int n, int h, int w, int relu_out, const void* mask_bf16, const void* add_bf16, ptta_stream_t stream);
/* the 32->32 TRANSPOSED stride-2 case (mode 2 of ptta_conv3x3: ConvTranspose2d(32,32,3,2,1,1) forward, Conv2d(s2) data gradient;
 * network_exp_msg_chn_adapt.py:276-283) on tcgen05.  h, w = INPUT size (w even); out / mask / add are [n, 2h, 2w, 32]. */
int ptta_pack_conv_weight_tc_t2(const void* wpack_bf16, void* wimage_bf16, ptta_stream_t stream);
int ptta_conv3x3_tc_t2(const void* in_bf16, void* out_bf16, const void* wimage_bf16, const float* bias, int n, int h, int w,
                       int relu_out, const void* mask_bf16, const void* add_bf16, ptta_stream_t stream);
/* timing experiments only: one eager step with a CUDA event after every kernel launch; prints the per-stream timeline */
int ptta_msgchn_trace_step(ptta_msgchn* engine, const float* image_raw, const float* img_scale3, const float* img_shift3,
                           const float* sparse_depth, float max_input_depth, float w_sd, float w_sm, float w_cos, ptta_stream_t stream);
/* weight gradient of a 3x3 stride-1 conv (autograd of the meta layer, network_exp_msg_chn_adapt.py:28-36) */
size_t ptta_conv3x3_wgrad_workspace_bytes(int n, int h, int w, int cin, int cout);
int ptta_conv3x3_wgrad(const void* in_bf16, const void* gout_bf16, float* dw, void* workspace,
                       int n, int h, int w, int cin, int cout,
                       int prologue, const float* pro_scale, const float* pro_shift, float slope, ptta_stream_t stream);
/* {1,2,3}-plane fp32 -> 32-channel stem conv (init.0 layers, :172,220), optional ReLU mask */
int ptta_stem_conv(const float* const* planes, const long long* batch_strides, const float* scale, const float* shift,
                   int cin, const float* weight, const float* bias, const void* mask_bf16, void* out_bf16,
                   int n, int h, int w, ptta_stream_t stream);
/* same operator with the weights ([32][cin][3][3]) and bias given as HOST arrays: they travel by value in the kernel parameters, so the
 * inner loop is FMAs with constant-bank operands only (what the engine uses for its frozen stems).  w must be even. */
int ptta_stem_conv_const(const float* const* planes, const long long* batch_strides, const float* scale, const float* shift,
                         int cin, const float* weight_host, const float* bias_host, const void* mask_bf16, void* out_bf16,
                         int relu_out, int n, int h, int w, ptta_stream_t stream);
/* 32 -> 1 conv (prdct.3, :289); weight is [9][32] fp32 */
int ptta_head_conv(const void* in_bf16, const float* weight_9x32, float bias, const float* add, float* out,
                   int n, int h, int w, int relu_in, int accumulate, ptta_stream_t stream);
/* same with the [9][32] weight given as a HOST array (by-value kernel parameters, constant-bank FMA operands) */
int ptta_head_conv_const(const void* in_bf16, const float* weight_host_9x32, float bias, const float* add, float* out,
                         int n, int h, int w, int relu_in, int accumulate, ptta_stream_t stream);
/* {1,2,3} -> 32 stem on tcgen05 (stem_tc_kernel: operand tiles built by the CUDA cores as bf16 head + remainder, six MMAs per 128 pixels);
 * weight: fp32 [32][cin][3][3] device, or NULL when image_scratch still holds the packed weights of an earlier call;
 * image_scratch: 4 096 bytes of device memory for the packed weights; any h, w */
int ptta_stem_conv_tc(const float* const* planes, const long long* batch_strides, const float* scale, const float* shift, int cin,
                      const float* weight, const float* bias, const void* mask_bf16, void* out_bf16, void* image_scratch, int relu_out,
                      int n, int h, int w, ptta_stream_t stream);
/* the same layer on tcgen05 (conv3x3_tc_head_kernel; the input must already hold ReLU(.) where the layer reads it through one):
 * pack: fp32 [9][32] device weights -> 9 216-byte weight image (bf16 head + bf16 remainder of every weight);
 * run: out[n][y][x] = bias [+ add[n][y][x]] + conv(in) ; w must be even */
int ptta_pack_head_weight_tc(const float* weight_9x32, void* image, ptta_stream_t stream);
int ptta_head_conv_tc(const void* in_bf16, const void* weight_image, float bias, const float* add, float* out, int n, int h, int w,
                      ptta_stream_t stream);
/* F.interpolate(scale_factor=2, bilinear, align_corners=True) (:201-209,493,500) and adjoints */
int ptta_up2_1ch(const float* a, const float* b, const float* c, float* out, int n, int h, int w, ptta_stream_t stream);
int ptta_up2_1ch_adjoint(const float* g_hi, float* g_lo, int n, int h, int w, int accumulate, ptta_stream_t stream);
int ptta_add_up2_c32(const void* x_bf16, const void* half_bf16, void* out_bf16, int n, int h, int w, ptta_stream_t stream);
int ptta_up2_c32_adjoint(const void* g_hi_bf16, void* g_lo_bf16, int n, int h, int w, int accumulate, ptta_stream_t stream);
/* nn.Linear (:1089-1098): C[M][N] = A[M][K] * B[N][K]^T + bias */
int ptta_gemm_bf16(const void* a, const void* b, void* c, const float* bias, long long m, int n, int k, ptta_stream_t stream);
/* the same on the tcgen05 tensor cores (TMA-fed, TMEM accumulators); needs N % 256 == 0 and K % 64 == 0 */
int ptta_gemm_bf16_tc(const void* a, const void* b, void* c, const float* bias, long long m, int n, int k, ptta_stream_t stream);
/* torch.optim.Adam over one flat fp32 buffer (src/tta_main.py:341-346,633); step is 1-based */
int ptta_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                   double lr, double beta1, double beta2, double eps, double weight_decay, int step, ptta_stream_t stream);
/* same update with the step counter (int, incremented by the call) and the hyper-parameters {lr, beta1, beta2, eps, weight_decay}
 * (doubles) in DEVICE memory, so the call can be captured into a CUDA graph and replayed */
int ptta_adam_flat_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, const double* hyper_dev,
                       int* step_dev, ptta_stream_t stream);
/* shared-model mode of the same update (ptta_comm, below): the flat gradient buffer is mean-all-reduced over the ranks inside the kernel
 * (ranks summed in rank order, bit-identical on all of them), the average is written back to grad, then the update runs.  xid: the
 * exchange id of the call within the step (all ranks issue the same sequence).  n <= the communicator's grad_floats. */
int ptta_adam_flat_dev_comm(float* param, float* grad, float* exp_avg, float* exp_avg_sq, long long n, const double* hyper_dev,
                            int* step_dev, ptta_comm* comm, int xid, ptta_stream_t stream);

/* ---- NLSPN non-local spatial propagation (SURVEY.md section 8 a20-a21) ----------------------------- */
/* DCN.modulated_deform_conv_forward / _backward, the reference's one native FFI
 * (external_src/NLSPN/src/model/deformconv/src/vision.cpp:6-13, modulated_deform_conv.h:10-87,
 * cuda/modulated_deform_conv_cuda.cu:19-290): fp32 NCHW, offset [N, 2*kh*kw, Ho, Wo] ordered (dh, dw) per tap,
 * mask [N, kh*kw, Ho, Wo], weight [C_out, C_in, kh, kw].  Implemented for what NLSPN calls: C_in = C_out = groups =
 * deformable_groups = 1, square odd kernel <= 7, stride 1, dilation 1 (3x3 pad 1 propagation, 1x1 pad 0 confidence
 * gather, nlspnmodel_adapt.py:300-304,332-336); anything else returns an error.  No columns buffer, no workspace.
 * backward: grad_input / grad_weight / grad_bias may be null (then not computed); grad_input is zero-filled here. */
int ptta_mdconv_forward(const float* input, const float* weight, const float* bias, const float* offset, const float* mask,
                        float* output, int n, int c_in, int h, int w, int c_out, int kh, int kw, int stride, int pad, int dil,
                        int groups, int deformable_groups, ptta_stream_t stream);
int ptta_mdconv_backward(const float* input, const float* weight, const float* offset, const float* mask, const float* grad_output,
                         float* grad_input, float* grad_offset, float* grad_mask, float* grad_weight, float* grad_bias,
                         int n, int c_in, int h, int w, int c_out, int kh, int kw, int stride, int pad, int dil,
                         int groups, int deformable_groups, ptta_stream_t stream);
/* NLSPN._get_offset_affinity (nlspnmodel_adapt.py:255-330; affinity 'TGASS', k_f = 3): offset_aff [N,24,H,W] is the output
 * of conv_offset_aff(guidance); confidence [N,1,H,W] or null (conf_prop off); legacy = the grid offset of :296-300.
 * Outputs offset [N,18,H,W] and aff [N,9,H,W] in the layout ptta_nlspn_propagate_* and ptta_mdconv_* take.
 * backward writes grad_offset_aff [N,24,H,W] and (zero-filled here, may be null) grad_confidence [N,1,H,W]. */
int ptta_nlspn_offset_affinity_forward(const float* offset_aff, const float* confidence, float aff_scale_const, int legacy,
                                       float* offset, float* aff, int n, int h, int w, ptta_stream_t stream);
int ptta_nlspn_offset_affinity_backward(const float* offset_aff, const float* confidence, float aff_scale_const, int legacy,
                                        const float* grad_offset, const float* grad_aff, float* grad_offset_aff, float* grad_confidence,
                                        int n, int h, int w, ptta_stream_t stream);
/* NLSPN.forward propagation loop (nlspnmodel_adapt.py:352-373): prop_time steps of
 *   feat = feat_fix > 0 ? feat_fix : feat;  feat = sum_k aff_k * bilinear(feat, p + grid_k + offset_k)
 * offset [N,18,H,W], aff [N,9,H,W] (after _get_offset_affinity), feat_* [N,1,H,W]; feat_fix may be null (preserve_input off).
 * `saved` (ptta_nlspn_saved_bytes) receives the blended input of every step (needed by backward); `list_feat`
 * (optional, [prop_time][N,H,W]) receives every step's output as the reference's list_feat does.
 * backward: gradient of the final feature only (the TTA loss reads nothing else); scratch = ptta_nlspn_backward_scratch_bytes. */
size_t ptta_nlspn_saved_bytes(int n, int h, int w, int prop_time);
size_t ptta_nlspn_backward_scratch_bytes(int n, int h, int w);
int ptta_nlspn_propagate_forward(const float* feat_init, const float* offset, const float* aff, const float* feat_fix, float* feat_out,
                                 float* saved, float* list_feat, int n, int h, int w, int prop_time, ptta_stream_t stream);
int ptta_nlspn_propagate_backward(const float* grad_out, const float* offset, const float* aff, const float* feat_fix, const float* saved,
                                  float* grad_feat_init, float* grad_offset, float* grad_aff, float* scratch,
                                  int n, int h, int w, int prop_time, ptta_stream_t stream);

/* the three TTA losses as stand-alone calls (src/loss_utils.py:116-169,624-638; src/external_model_adapt.py:371-441, incl. the
 * `loss_cos < 0.3 -> w_cos = 0` gate on the device).  emb / ref: bf16 [rows][dim].  The first five floats of `workspace` are
 * (loss, loss_sparse_depth, loss_smooth, loss_cos, w_cos_eff) after forward.  backward: g_pred fp32 [n,h,w], g_ref bf16 [rows][dim]. */
size_t ptta_tta_loss_workspace_bytes(int n, int h, int w, long long rows);
int ptta_tta_loss_forward(const float* pred, const float* image_raw, const float* sparse_depth, const float* validity,
                          float max_input_depth, const void* emb_bf16, const void* ref_bf16, long long rows, int dim,
                          float w_sparse_depth, float w_smoothness, float w_cos, void* workspace, int n, int h, int w,
                          ptta_stream_t stream);
int ptta_tta_loss_backward(const float* pred, const float* image_raw, const float* sparse_depth, const float* validity,
                           float max_input_depth, const void* emb_bf16, const void* ref_bf16, long long rows, int dim,
                           float w_sparse_depth, float w_smoothness, void* workspace, float grad_scale, float* g_pred,
                           void* g_ref_bf16, int n, int h, int w, ptta_stream_t stream);
/* gradient of the cosine loss with respect to `emb` (same workspace, after ptta_tta_loss_forward): needed when the proxy heads hold adapted
 * tensors (NLSPN adapt mode 'meta_bn' after convert_syncbn: src/nlspn_model_adapt.py:328-337 on SyncBatchNorm-converted BatchNorm1d) */
int ptta_tta_loss_backward_emb(const void* emb_bf16, const void* ref_bf16, long long rows, int dim, void* workspace, float gscale,
                               void* g_emb_bf16, int n, int h, int w, ptta_stream_t stream);
/* stage-2 loss of the source-domain preparation on stand-alone buffers: mean(2 - 2 cos(emb, ref)), no loss_cos gate
 * (src/external_model_adapt.py:524-540 `prepare_loss`); workspace as ptta_tta_loss_forward (float 0 = the loss), followed by
 * ptta_tta_loss_backward_emb for d loss / d emb. */
int ptta_cos_loss_forward(const void* emb_bf16, const void* ref_bf16, long long rows, int dim, void* workspace, int n, int h, int w,
                          ptta_stream_t stream);
/* EMA copy of a head tensor: target <- target * tau + source * (1 - tau) in the reference's operation order
 * (external_src/NLSPN/src/model/nlspnmodel_adapt.py:1314-1316 `_update_head`). */
int ptta_ema_update(float* target, const float* source, long long count, double tau, ptta_stream_t stream);

/* ---- general-channel convolutions of the NLSPN network (tcgen05, csrc/conv_gen.cuh) ------------------------------
 * external_src/NLSPN/src/model/nlspnmodel_adapt.py:384-448 (resnet34.layer1-4 = torchvision BasicBlock stacks, conv6,
 * dec5..dec2 ConvTranspose2d with skip concat, id/gd/cf_dec1) and the data gradients autograd runs for them.
 * kind: 0 Conv2d 3x3 s1 p1 | 1 Conv2d 3x3 s2 p1 | 2 ConvTranspose2d 3x3 s2 p1 op1 | 3 Conv2d 1x1 s2.
 * role: 0 forward (x0 [n,h,w,cin0] (+ x1 [n,h,w,cin1], the second half of a channel concat) -> out), 1 data gradient
 * (x0 = dL/d(layer output) -> out = dL/d(layer input) [n,h,w,cin0]; cin1 must be 0; has_short: kind 1 only, x1 = gradient
 * of the block's 1x1/s2 shortcut output, its weight packed behind the 3x3 one).  h, w = LAYER INPUT size.  All maps NHWC
 * bf16 with stored channel counts that are multiples of 64; weights are the reference's fp32 tensors (cin_w / cout_w real
 * channels, zero-padded to the stored counts).  ident_from >= 0: output channels >= ident_from copy the same input channel
 * (centre-tap identity; used to carry conv1_dep's 16 channels through the 48->48 meta conv, nlspnmodel_adapt.py:866-870). */
long long ptta_convg_packed_elems(int kind, int role, int cin0, int cin1, int cout, int has_short);
int ptta_convg_pack(int kind, int role, const float* weight, const float* weight_short, int cin_w, int cout_w,
                    int cin0, int cin1, int cout, int has_short, int ident_from, void* packed_bf16, ptta_stream_t stream);
int ptta_convg_run(int kind, int role, const void* x0_bf16, const void* x1_bf16, const void* packed_bf16, const float* bias,
                   void* out_bf16, int n, int h, int w, int cin0, int cin1, int cout, int has_short, ptta_stream_t stream);

/* host-only introspection of the K-item plan of a layer (CPU tests replay the implicit GEMM from it): header[16] = {n_items,
 * n_classes, th, tw, tiles_y, tiles_x, n_tiles, BN, halo, b_resident, n_a, n_b, in_parity, out_parity, n_out, halo_rev}, 4 x
 * {start, count, out_c, out_py} per class, then {c_inner, dx, dy, py, src, wsel, tap, k0} per item; returns the ints written */
int ptta_convg_plan_describe(int kind, int role, int n, int h, int w, int cin0, int cin1, int cout, int has_short, int* out,
                             int capacity);
/* mask 32: streamed weight tiles multicast over clusters of two CTAs (results unchanged; a tested option, off by default); mask 0: off.
 * Every other bit fails in this library: the work-skipping timing switches (1, 2, 4, 8, 16: results wrong by construction) and the cycle
 * stamps (64, read back through the two functions below) are compiled into the experiments build only (-DPTTA_EXPERIMENTS ->
 * lib/libptta_b200_experiments.so, used by tools/convg_experiment.py / convg_trace.py, never by the package): the product kernel
 * contains none of their branches. */
int ptta_convg_debug_set(int mask);
int ptta_convg_debug_read_ts(long long* out_host, int n);                /* experiments build only */
int ptta_convg_debug_read_cta(unsigned long long* out_host, int n);      /* experiments build only */
/* thin heads id_dec0 / gd_dec0 / cf_dec0 (nlspnmodel_adapt.py:430-448, 883-895) as ONE 16-output-channel conv over the concat
 * (x0 | x1): fp32 planar outputs through per-channel plane pointers (host arrays of n_real entries), activation per channel
 * (0 none, 1 LeakyReLU(0.2), 2 sigmoid).  Weights packed by ptta_convg_pack(kind 0, role 0, ..., cout = 16). */
int ptta_convg_run_thin(const void* x0_bf16, const void* x1_bf16, const void* packed_bf16, const float* bias, float* const* planes,
                        const long long* image_strides, const int* acts, int n_real, int n, int h, int w, int cin0, int cin1,
                        ptta_stream_t stream);

/* ---- channel-generic kernels of the NLSPN network (csrc/nlspn_net.cuh); NHWC bf16 maps [rows][c], c % 64 == 0 ------------- */
/* conv1_rgb + conv1_dep + LeakyReLU(0.2) (nlspnmodel_adapt.py:385-388, 866-867); image == NULL: the zero image of :907;
 * scale3 / shift3 (nullable): per-channel image normalisation x*scale+shift folded into the load (src/tta_main.py:595-604) */
int ptta_nl_stem(const float* image_nchw, const float* depth, const float* w_rgb, const float* b_rgb, const float* w_dep,
                 const float* b_dep, const float* scale3, const float* shift3, void* out_bf16_c64, int n, int h, int w,
                 ptta_stream_t stream);
/* merged batch: out [2n,h,w,64] = the n real images followed by their zero-image copies (same sparse depth), one launch */
int ptta_nl_stem_pair(const float* image_nchw, const float* depth, const float* w_rgb, const float* b_rgb, const float* w_dep,
                      const float* b_dep, const float* scale3, const float* shift3, void* out_bf16_c64, int n, int h, int w,
                      ptta_stream_t stream);
/* number of partial blocks the reductions below use: `partial` must hold 2 * c * blocks floats */
int ptta_nl_reduce_blocks(long long rows, int c);
/* train-mode BatchNorm statistics (batch mean, biased variance) -> mean, rstd, scale = gamma*rstd, shift = beta - mean*scale;
 * run_mean/run_var/num_batches_tracked (nullable): momentum update with the unbiased variance (BatchNorm1d of the heads) */
int ptta_nl_bn_stats(const void* x_bf16, long long ldx, long long rows, int c, const float* gamma, const float* beta, float eps,
                     float* partial, float* mean, float* rstd, float* scale, float* shift, float* run_mean, float* run_var,
                     long long* num_batches_tracked, float momentum, ptta_stream_t stream);
/* the same statistics for `groups` independent row ranges of rows_per_group rows each (real | zero-image halves of a merged
 * batch: each half is its own forward pass in the reference, nlspnmodel_adapt.py:866-914); outputs are [groups][c]; `partial` must
 * hold groups * 2 * c * ptta_nl_reduce_blocks(rows_per_group, c) floats.  ptta_nl_bn_act_grouped applies group g's vectors to its rows */
int ptta_nl_bn_stats_grouped(const void* x_bf16, long long ldx, long long rows_per_group, int groups, int c, const float* gamma,
                             const float* beta, float eps, float* partial, float* mean, float* rstd, float* scale, float* shift,
                             ptta_stream_t stream);
int ptta_nl_bn_act_grouped(const void* x_bf16, const float* scale, const float* shift, const void* res_bf16, long long ldr,
                           const float* rscale, const float* rshift, void* y_bf16, long long rows_per_group, int groups, int c, int act,
                           ptta_stream_t stream);
int ptta_nl_col_sums(const void* x_bf16, long long ldx, long long rows, int c, float* partial, float* sums, ptta_stream_t stream);
/* y = act(x*scale + shift [+ res | + res*rscale + rshift]); act: 0 none, 1 ReLU, 2 LeakyReLU(0.2) */
int ptta_nl_bn_act(const void* x_bf16, const float* scale, const float* shift, const void* res_bf16, long long ldr,
                   const float* rscale, const float* rshift, void* y_bf16, long long rows, int c, int act, ptta_stream_t stream);
/* g = (dy_a [+ dy_b]) * act'(y); dgamma = sum g*xhat, dbeta = sum g (nullable); dx = gamma*rstd*(g - mean(g) - xhat*mean(g*xhat));
 * gskip (nullable) receives g.  coef: 3*c floats of scratch. */
int ptta_nl_bn_backward(const void* dy_a, long long ld_a, const void* dy_b, long long ld_b, const void* y_bf16, int act,
                        const void* x_bf16, const float* mean, const float* rstd, const float* gamma, float* partial,
                        float* dgamma, float* dbeta, float* coef, void* dx_bf16, void* gskip_bf16, long long rows, int c,
                        ptta_stream_t stream);
/* shared-model mode (SyncBatchNorm over the ranks of `comm`): the same two calls with the per-channel sums exchanged through peer memory
 * inside the finalize kernel and added in rank order; count = rows x world.  xid: the exchange id of the call within the step.  The
 * backward's dgamma / dbeta stay the LOCAL sums (the gradient all-reduce averages them, as DDP does); dx uses the global means.  c <= 1024.
 * Every rank must issue the same sequence of exchanges, on one stream. */
int ptta_nl_bn_stats_comm(const void* x_bf16, long long ldx, long long rows, int c, const float* gamma, const float* beta, float eps,
                          float* partial, float* mean, float* rstd, float* scale, float* shift, float* run_mean, float* run_var,
                          long long* num_batches_tracked, float momentum, ptta_comm* comm, int xid, ptta_stream_t stream);
int ptta_nl_bn_backward_comm(const void* dy_a, long long ld_a, const void* dy_b, long long ld_b, const void* y_bf16, int act,
                             const void* x_bf16, const float* mean, const float* rstd, const float* gamma, float* partial,
                             float* dgamma, float* dbeta, float* coef, void* dx_bf16, void* gskip_bf16, long long rows, int c,
                             ptta_comm* comm, int xid, ptta_stream_t stream);
int ptta_nl_add3(const void* a, long long lda, const void* b, long long ldb, const void* c3, long long ldc, void* out, long long rows,
                 int c, ptta_stream_t stream);
/* output = clamp(y, min=0) (nlspnmodel_adapt.py:901) and its adjoint */
int ptta_nl_clamp0(const float* y, float* out, long long n, ptta_stream_t stream);
/* src/external_model_adapt.py:103-108: clamp(sparse_depth, 0, max_input_depth) */
int ptta_nl_clamp(const float* x, float* out, float lo, float hi, long long n, ptta_stream_t stream);
int ptta_nl_mask_pos(const float* g, const float* y, float* out, long long n, ptta_stream_t stream);
/* gradients of (pred_init, guide[8], confidence) through LeakyReLU / identity / sigmoid -> NHWC bf16 [n,h,w,64] (ch >= 10 zero) */
int ptta_nl_thin_grad_pack(const float* g_pred, const float* pred_init, const float* g_guide, const float* g_conf, const float* conf,
                           void* out_bf16_c64, int n, int h, int w, ptta_stream_t stream);
/* prop_layer.conv_offset_aff = Conv2d(8,24,3,1,1) in fp32 on planar maps (nlspnmodel_adapt.py:219-224,259); transposed != 0:
 * the data gradient ([n,24,h,w] -> [n,8,h,w]) */
int ptta_nl_conv8to24(const float* in, const float* weight, const float* bias, float* out, int n, int h, int w, int transposed,
                      ptta_stream_t stream);
/* weight gradient of the adapted Conv2d(48,48,3,1,1) meta layer (nlspnmodel_adapt.py:1370-1374) over 64-channel NHWC maps */
size_t ptta_nl_wgrad48_workspace_bytes(void);
int ptta_nl_wgrad48(const void* x_bf16_c64, const void* gout_bf16_c64, float* dw_48x48x3x3, void* workspace, int n, int h, int w,
                    ptta_stream_t stream);

/* evaluation metrics on the device (src/eval_utils.py:117-175 as used by src/tta_main.py:760-798): mask = gt > 0 and
 * min_depth <= gt <= max_depth; result5 (device) = {MAE [mm], RMSE [mm], iMAE [1/km], iRMSE [1/km], evaluated pixels} */
size_t ptta_eval_metrics_workspace_bytes(void);
int ptta_eval_metrics(const float* output_depth, const float* ground_truth, long long n, float min_depth, float max_depth,
                      void* workspace, float* result5, ptta_stream_t stream);

/* input stage (SURVEY.md 8f rank 2): src/data_utils.py:134-200 (load_image, load_depth_with_validity_map: depth = png / 256,
 * <= 0 -> 0, validity = depth > 0) + the crop of src/datasets.py:83-170, on decoded 8-bit RGB [n,h0,w0,3] and 16-bit depth [n,h0,w0]
 * payloads -> fp32 image NCHW in [0,255], depth and validity [n,1,h,w]; bit-exact with the numpy code */
int ptta_input_stage(const void* image_u8_hwc, const void* depth_u16, float* image_nchw, float* depth, float* validity, int n,
                     int h0, int w0, int y0, int x0, int h, int w, float depth_multiplier, ptta_stream_t stream);
/* On-device augmentations of the adaptation / preparation loops (src/transforms.py; the drop-in mirror with the reference's RNG draw
 * order is tta_depth_completion_b200/transforms.py).
 * ptta_augment_photometric: src/transforms.py:236-333 + :669-712 on an fp32 [N,3,H,W] image in [0,255]: uint8 truncation, per-sample
 * brightness / contrast / gamma / hue / saturation (the reference's order) as torchvision's tensor ops compute them (`_blend`,
 * `rgb_to_grayscale`, `adjust_gamma`, `adjust_hue`; every product and sum rounded separately, uint8 truncation after each transform),
 * `.float()`, additive noise (`noise`: fp32 [N,3,H,W] drawn by the caller -- torch.randn / torch.rand, so the generator contract holds --
 * added as x + spread * n, or spread * (n - 0.5) when noise_uniform), normalisation (norm_mode 0: none, 1: /255, 2: 2x/255-1,
 * 3: (x/255 - mean[c]) / std[c] with HOST arrays mean3 / std3).  Flag arrays: device uint8 [N] (NULL = transform not configured), factor
 * arrays: device fp32 [N].  quantize = 1 whenever any photometric transform is configured (the reference then casts to uint8 even for
 * samples that draw no transform).  workspace: 8 * n bytes, needed for the contrast transform (exact integer sum of the grey image).
 * ptta_augment_flip: src/transforms.py:990-1034, per-sample horizontal / vertical mirror of an fp32 [N,C,H,W] map (out != in). */
int ptta_augment_photometric(const float* image, float* out, int n, int h, int w, const unsigned char* do_brightness,
                             const float* f_brightness, const unsigned char* do_contrast, const float* f_contrast,
                             const unsigned char* do_saturation, const float* f_saturation, const unsigned char* do_gamma,
                             const float* f_gamma, const unsigned char* do_hue, const float* f_hue, const unsigned char* do_noise,
                             const float* noise, float noise_spread, int noise_uniform, int quantize, int norm_mode,
                             const float* mean3, const float* std3, void* workspace, ptta_stream_t stream);
int ptta_augment_flip(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_hflip,
                      const unsigned char* do_vflip, ptta_stream_t stream);
/* ptta_augment_rotate: src/transforms.py:406-423, 1036-1070 (torchvision functional.rotate, expand=False, fill=None = affine grid +
 * grid_sample with zero padding, align_corners=False).  theta_n_x_6: device fp32 [N][6], the 3 x 2 matrix torchvision multiplies its
 * base grid with (theta^T / (0.5 w, 0.5 h); x column first), prepared on the host as torchvision does.  mode 0 nearest, 1 bilinear.
 * ptta_augment_resize_crop: src/transforms.py:425-502, 1222-1283 (functional.resize to (resize_h, resize_w) >= (h, w), then the crop
 * [start_y, start_y + h) x [start_x, start_x + w)): device int32 [N] arrays; only the surviving h x w pixels are computed.
 * Both: fp32 [N,C,H,W], out != in, samples whose flag is clear are copied. */
/* ptta_augment_crop: src/transforms.py:337-383, 955-988 -- every sample cropped to the same (crop_h, crop_w) window at its own offset
 * (device int32 [N] arrays; the caller guarantees start + crop <= size, as torch.randint's bounds do); out is [N,C,crop_h,crop_w]. */
int ptta_augment_crop(const float* in, float* out, int n, int c, int h, int w, int crop_h, int crop_w, const int* start_y,
                      const int* start_x, ptta_stream_t stream);
/* ptta_augment_crop_pad: src/transforms.py:508-566, 1072-1135 with constant (zero) padding -- per sample the window
 * {start_y, start_x, crop_h, crop_w} is placed at {pad_top, pad_left} of an h x w map of zeros (device int32 [N][6] in that order). */
int ptta_augment_crop_pad(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_crop_pad,
                          const int* window_n_x_6, ptta_stream_t stream);
/* ptta_augment_remove_patches: src/transforms.py:625-652, 878-953 -- every selected pixel (`selected`: device uint8 [N,H,W], chosen by the
 * caller from the sample's non-zero pixels as the reference does, torch.randperm) erases the {ph, pw} patch around it (device int32 [N][2], odd). */
int ptta_augment_remove_patches(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_remove,
                                const unsigned char* selected, const int* patch_n_x_2, ptta_stream_t stream);
/* ptta_augment_resize_pad: src/transforms.py:578-622, 1137-1220 -- per sample a reduction to {resize_h, resize_w} <= (h, w) placed at {pad_top,
 * pad_left} of an h x w map of zeros (device int32 [N][4] in that order); nearest or bilinear WITHOUT anti-aliasing (torchvision 0.10.1, the
 * release the reference pins; later releases filter a bilinear reduction by default). */
int ptta_augment_resize_pad(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_resize_pad,
                            const int* geometry_n_x_4, int mode, ptta_stream_t stream);
/* ptta_augment_divide_samples: src/transforms.py:1274-1275 (`resize_scaling_depth`) -- in place, data[n][:] /= divisor[n] (IEEE fp32 division)
 * for the samples whose flag is set; the caller passes float32(r_width / n_width) of the resize-and-crop draw. */
int ptta_augment_divide_samples(float* data, int n, long long per_sample, const unsigned char* do_divide, const float* divisor_n, ptta_stream_t stream);
int ptta_augment_rotate(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_rotate,
                        const float* theta_n_x_6, int mode, ptta_stream_t stream);
int ptta_augment_resize_crop(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_resize,
                             const int* resize_h, const int* resize_w, const int* start_y, const int* start_x, int mode,
                             ptta_stream_t stream);

/* Host-side PNG decoding (no device work; plain host pointers, e.g. pinned staging memory): replaces PIL on the reference's loader path --
 * `np.asarray(Image.open(path).convert('RGB'))` (src/data_utils.py:134-165) and `np.array(Image.open(path))` of the 16-bit depth maps
 * (src/data_utils.py:167-234).  Container parsing with CRC check, zlib inflate, the five scanline filters, colour-type conversion as
 * convert('RGB') does it (alpha dropped, grey replicated, palette looked up).  8- and 16-bit non-interlaced files; anything else fails
 * with a message.  ptta_png_info: channels = 3 for palette files; bit_depth 8 or 16. */
int ptta_png_info(const void* file_bytes, size_t n, int* width, int* height, int* channels, int* bit_depth);
int ptta_png_decode_rgb8(const void* file_bytes, size_t n, unsigned char* out_hwc, size_t out_bytes);
int ptta_png_decode_gray16(const void* file_bytes, size_t n, unsigned short* out_hw, size_t out_bytes);

/* ---- MSG-CHN ProxyTTA engine ------------------------------------------------------------------- */
/* prepare_mode: the reference's string, e.g. "meta_selfsup_seq_2layers_ema" (network_exp_msg_chn_adapt.py:1022-1087) */
int ptta_msgchn_create(ptta_msgchn** out, int n, int h, int w, const char* prepare_mode);
void ptta_msgchn_destroy(ptta_msgchn* e);
/* dispatch options (results stay right for every value; used by the parity tests to run ALL kernel families at every size):
 * "tc_min_pixels" / "tc_s2_min_pixels" / "tc_t2_min_pixels": smallest map (N*H*W of the INPUT) the stride-1 / stride-2 /
 * transposed tcgen05 convs take (0 = always),
 * "tc_enabled" 0/1, "two_streams" 0/1, "fuse_dec_sums" 0/1; "trainable_head" / "skip_dec3": see the preparation steps below.
 * Unknown names fail. */
/* ---- shared-model mode (BASELINE.json configs[4]; the reference: DDP + SyncBatchNorm, src/msg_chn_model_adapt.py:480,555-556) ----
 * One communicator per rank: a device block mapped into every peer through CUDA IPC.  With a communicator set, the engine's
 * train-mode BatchNorm layers take their statistics over ALL ranks (forward sums and backward sums exchanged through peer memory
 * inside the finalize kernels) and the Adam step first mean-all-reduces the flat adapted-gradient buffer (one fused kernel, ranks
 * summed in rank order: bit-identical replicas).  No NCCL call on the path; the step stays capturable in one CUDA graph.
 * Train-mode BatchNorm sums: exchanged inside bn_finalize / bn_bwd_finalize.  Host protocol: create -> local_handle -> exchange the handles (any transport, e.g. torch.distributed.all_gather_object) ->
 * open_peers -> ptta_msgchn_set_comm. */
int ptta_comm_create(ptta_comm** out, int rank, int world, long long grad_floats);
int ptta_comm_handle_bytes(void);
int ptta_comm_local_handle(ptta_comm* c, void* handle_out);
int ptta_comm_open_peers(ptta_comm* c, const void* handles_world_x_bytes);
int ptta_comm_error(ptta_comm* c);      /* 0 = fine; k > 0 = exchange k-1 timed out waiting for a peer (~4 s): results are void */
void ptta_comm_destroy(ptta_comm* c);
/* exchanges one step may use (exchange ids 0 .. max-1) */
int ptta_comm_max_exchanges(void);
/* end of a step driven through the ptta_*_comm entry points: the next step's exchanges use the next tag (the MSG-CHN engine does this
 * inside its Adam step) */
int ptta_comm_advance(ptta_comm* c, ptta_stream_t stream);
int ptta_msgchn_set_comm(ptta_msgchn* e, ptta_comm* c);
int ptta_msgchn_set_option(ptta_msgchn* e, const char* name, long long value);
size_t ptta_msgchn_workspace_bytes(const ptta_msgchn* e);
int ptta_msgchn_bind_workspace(ptta_msgchn* e, void* workspace, size_t bytes, ptta_stream_t stream);
/* bind one state-dict entry (fp32, or int64 for num_batches_tracked) by its reference key; also
 * "grad/<key>", "adam_m/<key>", "adam_v/<key>" for the adapted tensors. Pointers are not owned. */
int ptta_msgchn_set_tensor(ptta_msgchn* e, const char* key, void* device_ptr, long long numel);
/* number / names of state-dict keys the engine requires (for error reporting and tests) */
int ptta_msgchn_num_keys(const ptta_msgchn* e);
const char* ptta_msgchn_key(const ptta_msgchn* e, int i);
/* (re)build the bf16 operand copies: all layers (+ cached zero-image rgb_encoder features) or only the adapted meta layer */
int ptta_msgchn_pack_weights(ptta_msgchn* e, ptta_stream_t stream);
int ptta_msgchn_pack_adapted(ptta_msgchn* e, ptta_stream_t stream);
/* ExternalModel_Adapt.forward (src/external_model_adapt.py:82-114) -> network_adapt.forward
 * (network_exp_msg_chn_adapt.py:337-557).  image: fp32 NCHW; the network sees image*img_scale[c]+img_shift[c].
 * img_scale / img_shift are HOST arrays of 3 floats.  training != 0 also runs the zero-image branch and the proxy heads. */
int ptta_msgchn_forward(ptta_msgchn* e, const float* image, const float* img_scale, const float* img_shift,
                        const float* sparse_depth, float max_input_depth, int training, ptta_stream_t stream);
/* ExternalModel_Adapt.compute_loss(loss_type='adapt') -> adapt_loss (src/external_model_adapt.py:371-441) on the
 * outputs of the last training forward; results stay on the device (ptta_msgchn_read_losses syncs). */
int ptta_msgchn_loss(ptta_msgchn* e, const float* image_raw, const float* sparse_depth, const float* validity,
                     float max_input_depth, float w_sparse_depth, float w_smoothness, float w_cos, ptta_stream_t stream);
int ptta_msgchn_read_losses(ptta_msgchn* e, float* out5 /* loss, sparse, smooth, cos, w_cos_eff */, ptta_stream_t stream);
/* loss.backward() restricted to what the adapted tensors need (src/tta_main.py:631-632) */
int ptta_msgchn_backward(ptta_msgchn* e, float grad_scale, ptta_stream_t stream);
/* the same in two halves, for autograd integration: loss -> ("g_output" fp32 [N,H,W], "g_ref" bf16 [R,512]),
 * then ("g_output", "g_ref") -> gradients of the adapted tensors ("grad/<key>" buffers) */
int ptta_msgchn_loss_backward(ptta_msgchn* e, float grad_scale, ptta_stream_t stream);
int ptta_msgchn_network_backward(ptta_msgchn* e, ptta_stream_t stream);
/* optimizer.step() (src/tta_main.py:633) + repack of the adapted bf16 operands */
/* hyper-parameters are doubles (torch derives 1-beta and the bias corrections in double); step_count < 0 keeps the device-side count */
int ptta_msgchn_set_adam(ptta_msgchn* e, double lr, double beta1, double beta2, double eps, double weight_decay, int step_count, ptta_stream_t stream);
int ptta_msgchn_adam_step(ptta_msgchn* e, ptta_stream_t stream);
/* the whole per-frame step, src/tta_main.py:583-633: outlier removal, forward, loss, backward, Adam */
int ptta_msgchn_tta_step(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift,
                         const float* sparse_depth, float max_input_depth,
                         float w_sparse_depth, float w_smoothness, float w_cos, ptta_stream_t stream);
/* same step captured once into a CUDA graph and replayed (inputs are read from the same device buffers each launch) */
int ptta_msgchn_tta_step_graph(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift,
                               const float* sparse_depth, float max_input_depth,
                               float w_sparse_depth, float w_smoothness, float w_cos, ptta_stream_t stream);
/* ---- source-domain preparation steps (SURVEY.md section 8 f3; the reference: src/init_main.py:448-572, src/head_main.py:415-541) ----
 * The training forward's `training` argument is a mode: 0 eval, 1 train with the zero-image branch and the proxy heads (TTA and
 * stage 2), 2 train WITHOUT them (stage 1: network_exp_msg_chn_adapt.py:559-607, real branch only, meta BatchNorm in train mode).
 * Stage 1 (meta-layer initialisation, supervised): forward(mode 2) -> l2_loss = MsgChnModel_Adapt.compute_loss(loss_type='pretrain')
 * (src/msg_chn_model_adapt.py:224-264: ground truth clamped to [0, max_predict_depth], validity = gt > 0, per-image masked MSE, batch
 * mean) -> l2_loss_backward -> network_backward -> adam_step; ptta_msgchn_init_step runs the five in one call.
 * Stage 2 (predictor head, engine option "trainable_head" = 1 before the workspace is bound: Adam then steps pred.{0,1,3}.* instead of
 * the meta layer): forward(mode 1) -> ema_update_head (proj_t <- tau proj_t + (1 - tau) proj, network_exp_msg_chn_adapt.py:701-703) ->
 * cos_loss = prepare_loss (src/external_model_adapt.py:524-540, no loss_cos gate) -> cos_loss_backward -> head_backward (weight / bias gradients of pred.0 and
 * pred.3 through ptta_gemm_tn_bf16_tc, BatchNorm1d affine gradients; proj's output is detached, :692) -> adam_step;
 * ptta_msgchn_head_step runs them in one call.  Option "skip_dec3" = 1 leaves out decoder 3 (stage 2 never reads the prediction).
 * H and W must be multiples of 16 (the reference pads in 'adapt' mode only). */
int ptta_msgchn_l2_loss(ptta_msgchn* e, const float* ground_truth, float max_predict_depth, ptta_stream_t stream);
int ptta_msgchn_l2_loss_backward(ptta_msgchn* e, float grad_scale, ptta_stream_t stream);
int ptta_msgchn_init_step(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift, const float* sparse_depth,
                          const float* ground_truth, float max_input_depth, float max_predict_depth, ptta_stream_t stream);
/* the same two steps captured once into a CUDA graph and replayed (inputs copied into engine-owned staging buffers inside the call, so a
 * fresh tensor may be passed every step; needs a non-default stream) */
int ptta_msgchn_init_step_graph(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift, const float* sparse_depth,
                                const float* ground_truth, float max_input_depth, float max_predict_depth, ptta_stream_t stream);
int ptta_msgchn_head_step_graph(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift,
                                const float* sparse_depth, float max_input_depth, ptta_stream_t stream);
int ptta_msgchn_cos_loss(ptta_msgchn* e, ptta_stream_t stream);
int ptta_msgchn_ema_update_head(ptta_msgchn* e, double tau, ptta_stream_t stream);
int ptta_msgchn_cos_loss_backward(ptta_msgchn* e, float grad_scale, ptta_stream_t stream);      /* -> "g_emb" (bf16 [R,512]) */
int ptta_msgchn_head_backward(ptta_msgchn* e, ptta_stream_t stream);                             /* "g_emb" -> "grad/pred.*" */
int ptta_msgchn_head_step(ptta_msgchn* e, const float* image_raw, const float* img_scale, const float* img_shift, const float* sparse_depth,
                          float max_input_depth, ptta_stream_t stream);
/* C[m][n] (fp32) = A[rows][m]^T B[rows][n] (bf16, row-major): the weight gradient of a Linear layer, dW[out][in] = sum_r dY[r][out] X[r][in]
 * (torch: `grad_output.t().mm(input)` inside loss.backward(), src/head_main.py:479), tcgen05 with MN-major operands and a split over the
 * rows; m % 128 == 0, n % 256 == 0; workspace: ptta_gemm_tn_workspace_bytes (0 = unsupported shape). */
size_t ptta_gemm_tn_workspace_bytes(long long rows, int m, int n);
int ptta_gemm_tn_bf16_tc(const void* a_bf16, const void* b_bf16, float* c, void* workspace, long long rows, int m, int n, ptta_stream_t stream);
/* named access to engine-owned tensors ("output", "emb", "ref", "filtered_depth", "filtered_validity", any
 * activation by its debug name). dtype: 0 fp32, 1 bf16. dims: up to 4 (NHWC for maps). */
int ptta_msgchn_get_tensor(ptta_msgchn* e, const char* name, void** ptr, int* dtype, long long* dims4);
int ptta_msgchn_num_tensors(const ptta_msgchn* e);
const char* ptta_msgchn_tensor_name(const ptta_msgchn* e, int i);
/* number of kernels launched by this engine since creation (for bench.py's gpu_launches) */
long long ptta_msgchn_launch_count(const ptta_msgchn* e);

#ifdef __cplusplus
}
#endif
#endif
