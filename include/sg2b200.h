/*
 * sg2b200 — C ABI of the B200-native (sm_100a) StackGAN-v2 train-step kernels.
 *
 * The reference (smallflyingpig/speech-to-image-translation-without-text) has no FFI: its hot path is
 * torch.nn modules in StackGAN_v2/model.py that dispatch to cuDNN/cuBLAS. Each entry point below replaces
 * the library call(s) that one reference construct triggers; the reference file:line is cited per function.
 * Every pointer is a raw CUDA device pointer owned by the caller (PyTorch's caching allocator); `stream` is a
 * cudaStream_t passed as void*. All functions return 0 on success, a negative SG2_E* code for a rejected shape,
 * or a positive cudaError_t. Nothing here allocates, synchronises, or falls back to the CPU.
 *
 * Internal activation layout: NHWC, bf16.  Weight packs: bf16, see sg2_pack_weights.
 */
#ifndef SG2B200_H
#define SG2B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SG2_EINVAL (-1)  /* unsupported shape / argument */
#define SG2_EDRIVER (-2) /* cuTensorMapEncodeTiled unavailable or failed */
#define SG2_ENOFUSE (-3) /* the requested epilogue fusion is not possible for this shape: call the separate kernel */

/* Convolution kinds on the path. */
enum {
  SG2_CONV3x3 = 0,   /* conv3x3 s1 p1, no bias            model.py:125-128 */
  SG2_UPCONV3x3 = 1, /* nearest 2x upsample + conv3x3     model.py:133-140 (nn.Upsample folded into addressing) */
  SG2_CONV4x4S2 = 2, /* conv4x4 s2 p1, no bias            model.py:369-398 */
  SG2_GEMM = 3,      /* 1x1 / plain matmul                model.py:179, 217 */
  SG2_STEM4x4 = 4    /* pack-only: conv4x4 s2 on 3 channels as a K=48(->64) GEMM over sg2_stem_im2col rows, model.py:383 */
};
enum { SG2_ACT_NONE = 0, SG2_ACT_GLU = 1, SG2_ACT_LRELU = 2 };
enum { SG2_OUT_BF16 = 0, SG2_OUT_F32_ATOMIC = 1, SG2_OUT_F32_STORE = 2 };

int sg2_version(void);
const char* sg2_last_error(void);
/* Data-parallel runs: leave `n_sms` SMs out of the persistent (one CTA per SM) convolution grids so that NCCL's all-reduce
 * CTAs (trainer.py:165-171's DataParallel gradient exchange, here one ncclAllReduce per gradient bucket slice) can run
 * beside them. 0 (default): use every SM. Process-wide. */
int sg2_set_sm_reserve(int n_sms);
/* CTA-pair (cta_group::2) gather kernels on (1) / off (0: their layers run on the cluster / plain gather kernels) /
 * as the environment says (-1, default: SG2_PAIR, SG2_PAIR_WGRAD; on). Process-wide. The data-parallel trainer switches
 * them off unless SG2_PAIR is set: every multi-GPU configuration of the round was validated and measured that way. */
int sg2_set_pair_kernels(int on);

/* ---- weights ------------------------------------------------------------------------------------------
 * fp32 OIHW master weights (the nn.Conv2d .weight the optimiser owns) -> bf16 operand packs.
 *   wpk  : fprop operand  [groups][Cout][taps][Cin]      wpkT : dgrad operand [groups'][Cin][taps'][Cout]
 *   CONV3x3   wpk [1][Cout][9][Cin]   wpkT [1][Cin][9][Cout]
 *   UPCONV3x3 wpk [4][Cout][4][Cin]   wpkT [1][Cin][16][Cout]   (3x3 taps pre-summed per output parity)
 *   CONV4x4S2 wpk [1][Cout][16][Cin]  wpkT [4][Cin][4][Cout]
 *   GEMM      wpk [Cout][Cin]         wpkT [Cin][Cout]
 * Cout_pad/Cin_pad >= Cout/Cin give the padded operand extents (zero filled). Either output may be NULL.
 * src_ohwi / dst_ohwi = 1: the fp32 master (gradient) is stored [Cout][kh][kw][Cin] instead of OIHW — the layout the
 * fused trainer keeps its flat parameter buckets in, where the CONV3x3 / CONV4x4S2 fprop operand is a plain bf16 cast
 * of the master (written by sg2_adam_ema) and sg2_conv_wgrad accumulates straight into the gradient bucket. */
int sg2_pack_weights(int kind, const float* w, void* wpk, void* wpkT, int Cout, int Cin, int Cout_pad,
                     int Cin_pad, int src_ohwi, void* stream);
/* dgrad operand from the bf16 fprop operand (CONV3x3 / CONV4x4S2 / GEMM, unpadded): per-tap [Cout][Cin] transpose. */
int sg2_pack_transpose(int kind, const void* wpk, void* wpkT, int Cout, int Cin, void* stream);
/* dwpk [Cout_pad][jobs][Cin_pad] fp32 (what sg2_conv_wgrad accumulates) -> OIHW fp32 gradient (+= if accumulate). */
int sg2_unpack_wgrad(int kind, const float* dwpk, float* grad, int Cout, int Cin, int Cout_pad, int Cin_pad,
                     int accumulate, int dst_ohwi, void* stream);

/* ---- convolutions (tcgen05 implicit GEMM, TMA operands) ------------------------------------------------
 * B,H,W,Cin are the FORWARD input extents of the layer; Cout its output channels. Replaces cuDNN fprop /
 * dgrad / wgrad behind nn.Conv2d (+ nn.Upsample) at model.py:125-140, 358-398.
 *   fprop : x [B][H][W][Cin] -> y  (CONV3x3: [B][H][W][Cout]; UPCONV3x3: [B][2H][2W][Cout]; CONV4x4S2: [B][H/2][W/2][Cout])
 *   dgrad : dy (shape of y) -> dx [B][H][W][Cin]
 *   wgrad : dwpk[Cout][jobs][Cin] += dy^T (x) im2col(x)   (fp32, red.global.add)
 * out_mode: SG2_OUT_BF16 store, SG2_OUT_F32_ATOMIC (split-K accumulate into a zeroed fp32 buffer), SG2_OUT_F32_STORE.
 * stats (fprop, optional): fp64 [2][Cout], += per-channel sum and sum of squares of the bf16 outputs, computed in the
 * epilogue from the TMEM accumulators (the BatchNorm batch statistics, consumed by sg2_bn_act_fwd). stats_groups > 1:
 * the batch is `stats_groups` equal sub-batches with separate statistics, stats [groups][2][Cout]; returns SG2_ENOFUSE
 * when a pixel tile of this shape would straddle two sub-batches (use sg2_bn_stats then).
 * act (fprop): 0, or SG2_ACT_LRELU applied in the epilogue (layers without BatchNorm: the D stems, model.py:383-384).
 * bias9 (fprop, CONV3x3, optional): fp32 [B][9][Cout] added to the accumulators before statistics / store; row
 * (ry*3+rx) applies to the pixels of border class ry = {top row, interior, bottom row} x rx = {left, interior, right}
 * (see sg2_joint_bias: the broadcast c_code channels of a jointConv folded into a per-sample bias). */
int sg2_conv_fprop(int kind, const void* x, const void* wpk, void* y, int out_mode, int B, int H, int W, int Cin,
                   int Cout, int splitk, double* stats, int stats_groups, int act, const float* bias9, void* stream);
/* dgrad epilogue operand (optional): epi_src has the shape of dx (bf16). SG2_EPI_ADD: dx = dgrad + epi_src (the skip
 * branch of a ResBlock's backward, model.py:166-169). SG2_EPI_LRELU_MASK: dx = dgrad * (epi_src > 0 ? 1 : 0.2), the
 * backward of the LeakyReLU(0.2) that produced epi_src (D stems, model.py:383-384). Returns SG2_ENOFUSE for shapes that
 * run on the gather kernel or split K (apply sg2_add_bf16 / sg2_lrelu_bwd afterwards instead). */
enum { SG2_EPI_NONE = 0, SG2_EPI_ADD = 1, SG2_EPI_LRELU_MASK = 2 };
int sg2_conv_dgrad(int kind, const void* dy, const void* wpkT, void* dx, int out_mode, int B, int H, int W, int Cin,
                   int Cout, int splitk, const void* epi_src, int epi_mode, void* stream);
/* wgrad, deterministic mode (partials != NULL): every pixel split (gather kernel: `splitk` splits; tile kernel: its CTA
 * lanes) STORES its partial result into its own slab partials[s][Cout][jobs][Cin]; sum them in slab order with
 * sg2_reduce_slabs. sg2_conv_wgrad_slabs returns how many slabs this shape / splitk writes (>= 1; negative = error).
 * partials == NULL: fp32 red.global.add straight into dwpk (faster for large weights with few splits, summation order
 * not reproducible run to run). */
int sg2_conv_wgrad(int kind, const void* x, const void* dy, float* dwpk, int B, int H, int W, int Cin, int Cout,
                   int splitk, float* partials, void* stream);
int sg2_conv_wgrad_slabs(int kind, int B, int H, int W, int Cin, int Cout, int splitk);
/* dst[i] (=|+=) sum_s parts[s * slab + i], s in order (n, slab multiples of 4; 16-byte aligned pointers). */
int sg2_reduce_slabs(const float* parts, int nslabs, long long n, long long slab, float* dst, int accumulate,
                     void* stream);
/* Split-K fprop / dgrad, deterministic mode: sg2_conv_fprop / sg2_conv_dgrad with SG2_OUT_F32_STORE and splitk > 1 store
 * split s into slab s (y + s * B*Ho*Wo*Cout floats); this sums the slabs in order, applies the optional dgrad epilogue
 * operand (SG2_EPI_*), rounds to bf16 [P][C] and (stats != NULL) accumulates the BatchNorm statistics of the rounded
 * values. nsplit == 1: a plain fp32 -> bf16 conversion (+ statistics). */
int sg2_splitk_finish(const float* parts, int nsplit, long long slab, void* y, long long P, int C, int groups,
                      double* stats, const void* epi_src, int epi_mode, void* stream);

/* ---- Inception-v3 scorer (model.py:17-109: torchvision Inception3 in eval mode, run at trainer.py:563-565) ---------
 * Every BasicConv2d (conv without bias, BatchNorm2d(eps=0.001) on running statistics, ReLU) is one convolution with a
 * folded bias and ReLU in the epilogue. NHWC bf16 activations; an Inception block's branches write straight into their
 * channel slice of the block output (no concat).
 * sg2_conv2d_fprop: y = relu?(conv(x, w) + bias) on the tcgen05 gather kernel; kh x kw <= 32 taps, stride 1 or 2, zero
 *   padding ph / pw on both sides of each axis (0 = a "valid" convolution). x: the Cin channels of an NHWC tensor whose
 *   pixel stride is x_ctot channels (a channel slice: pass the slice's first element); y: [B][Ho][Wo] pixels of y_ctot
 *   channels, Cout of them written. wpk: bf16 [Cout][kh][kw][Cin]; bias: fp32 [Cout] (may be NULL). Cin % 16 == 0,
 *   Cout, x_ctot, y_ctot % 8 == 0.
 * sg2_conv2d_plan: the tiling the same call would use, computed from shapes: out[8] = {issued MMA rows, useful rows
 *   (output pixels), issued MMA columns, BN, BK, tile width, tile height, images per tile}. */
int sg2_conv2d_fprop(const void* x, int x_ctot, const void* wpk, const float* bias, void* y, int y_ctot, int B, int H,
                     int W, int Cin, int Cout, int kh, int kw, int stride, int ph, int pw, int relu, void* stream);
int sg2_conv2d_plan(int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride, int ph, int pw, long long* out);
/* sg2_inception_stem: img NCHW fp32 [B][3][S][S] in [-1, 1] -> col [B][149][149][32] bf16, the im2col rows of
 *   Conv2d_1a_3x3 (3x3 s2 p0, K = 27 = (ky, kx, c), zero padded to 32) of the preprocessed image: x * 0.5 + 0.5, per-channel
 *   (x - mean) / std with the ImageNet mean / std, bilinear resize to 299 x 299 (align_corners=False). No 299^2 image. */
int sg2_inception_stem(const float* img, void* col, int B, int S, void* stream);
/* max-pool 3x3 s2 p0 (y may be a channel slice: y_ctot channels per pixel); avg-pool 3x3 s1 p1 count_include_pad=True;
 * C % 8 == 0. */
int sg2_maxpool3s2(const void* x, void* y, int y_ctot, int B, int H, int W, int C, void* stream);
int sg2_avgpool3s1(const void* x, void* y, int B, int H, int W, int C, void* stream);
/* out [B][C] fp32 = mean over the HW pixels of x [B][HW][C] bf16 (pool3: adaptive 8x8 average, summed in pixel order) */
int sg2_global_avg(const void* x, float* out, int B, int HW, int C, void* stream);
/* row softmax, fp32 [M][N] -> [M][N] */
int sg2_softmax_rows(const float* x, float* y, int M, int N, void* stream);

/* ---- jointConv with the broadcast c_code folded away (NEXT_STAGE_G, model.py:274-279) ---------------------------
 * conv3x3(cat(c (x) 1, h)) = conv3x3_h(h) + bias9[b][border class][o]: the c_code channels are constant over the image,
 * so their share is a per-sample bias that depends only on which taps fall inside the image (sg2_conv_fprop's bias9).
 * w: the fp32 master of the FULL weight, element (o, e, tap) at w[o*so + e*se + tap*st]; the c_code channels are the
 * first E input channels (model.py:277 puts c_code first).
 *   sg2_joint_bias     : c [B][E] -> bias9 [B][9][Cout]
 *   sg2_joint_tap_sums : dy [B][H][W][Cout] bf16 -> S [B][9 taps][Cout] = sum of dy over the pixels where the tap is
 *                        inside the image (R: fp64 [B][9][Cout] ZEROED workspace). Two launches.
 *   sg2_joint_c_bwd    : dw[o][e][tap] (=|+=) sum_b c[b][e] S[b][tap][o] (same strides as w; NULL to skip);
 *                        dc[b][e] += sum_{o,tap} w[o][e][tap] S[b][tap][o] (NULL to skip). One launch each. */
int sg2_joint_bias(const float* c, const float* w, long long so, long long se, long long st, float* bias9, int B, int E,
                   int Cout, void* stream);
int sg2_joint_tap_sums(const void* dy, double* R, float* S, int B, int H, int W, int Cout, void* stream);
int sg2_joint_c_bwd(const float* S, const float* c, const float* w, long long so, long long se, long long st, float* dc,
                    float* dw, int dw_accumulate, int B, int E, int Cout, void* stream);

/* ---- BatchNorm (+ GLU / LeakyReLU(0.2) / residual) on [P pixels][C channels] bf16 ---------------------
 * nn.BatchNorm2d/1d train mode (model.py:137,147,158,161,218,361,372,387-394): batch mean, biased variance,
 * eps, momentum; running_var gets the unbiased variance; num_batches_tracked += 1.
 * stats: fp64 [2][C] per-channel sum / sum of squares, accumulated (+=) into a ZEROED workspace either by the conv
 * epilogue (sg2_conv_fprop), by sg2_f32_to_bf16_stats (split-K accumulators, fc outputs) or by sg2_bn_stats.
 * groups > 1: the P rows are `groups` consecutive equal slabs (sub-batches), each normalised on its OWN statistics
 * (stats [groups][2][C], mean/rstd [groups][C], sums [groups][2][C]) — the same arithmetic as `groups` separate
 * nn.BatchNorm calls (train_Dnet's real / wrong / fake passes, trainer.py:390-392); running statistics are updated
 * once per group in order, num_batches_tracked += groups, dgamma/dbeta sum over the groups. */
int sg2_bn_stats(const void* x, long long P, int C, int groups, double* stats, void* stream);
int sg2_f32_to_bf16_stats(const float* x, void* y, long long P, int C, int groups, double* stats, void* stream);
int sg2_bn_eval_prepare(const float* running_mean, const float* running_var, float eps, float* mean, float* rstd,
                        int C, void* stream);
/* out = act(bn(x)) (+ residual, ACT_NONE only). GLU (model.py:112-122) halves the channel count.
 * train: stats != NULL -> mean/rstd are derived in-kernel, written to mean/rstd (saved for backward) and the running
 * statistics are updated.  eval: stats == NULL, mean/rstd are inputs.  mean == NULL: no BatchNorm (D stem). */
int sg2_bn_act_fwd(const void* x, const double* stats, float* mean, float* rstd, const float* gamma, const float* beta,
                   const void* residual, void* out, long long P, int C, int groups, int act, float eps, float momentum,
                   float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
/* dx (shape of x) from dout (shape of out); dgamma/dbeta (=|+=). sums: fp64 [2][C] ZEROED workspace. Two launches. */
int sg2_bn_act_bwd(const void* x, const void* dout, const float* mean, const float* rstd, const float* gamma,
                   const float* beta, double* sums, void* dx, float* dgamma, float* dbeta, int accumulate,
                   long long P, int C, int groups, int act, void* stream);
int sg2_lrelu_bwd(const void* x, const void* dout, void* dx, long long n, void* stream);
int sg2_add_bf16(const void* a, const void* b, void* out, long long n, void* stream);
int sg2_f32_to_bf16(const float* in, void* out, long long n, void* stream);
int sg2_bf16_to_f32(const void* in, float* out, long long n, void* stream);   /* n % 4 == 0 (gradient slices on the bf16 wire) */

/* ---- broadcast c_code concat (model.py:274-277, 431-434): out[b,y,x,:] = (c[b,:E] | h[b,y,x,:Ch]) -------- */
int sg2_concat_c(const float* c, const void* h, void* out, int B, int HW, int E, int Ch, void* stream);
int sg2_concat_c_bwd(const void* dcat, void* dh, float* dc /* += */, int B, int HW, int E, int Ch, void* stream);

/* ---- image heads (model.py:287-298) and D stems (model.py:383) --------------------------------------------- */
int sg2_head_tanh_fwd(const void* y /* [P][CP] bf16 */, float* img /* NCHW fp32 */, int B, int HW, int CP, void* stream);
int sg2_head_tanh_bwd(const float* dimg, const float* img, void* dy, int B, int HW, int CP, void* stream);
int sg2_stem_im2col(const float* img /* NCHW fp32 [B][3][S][S] */, void* col /* [B*(S/2)^2][64] bf16 */, int B, int S,
                    void* stream);
int sg2_stem_col2im(const void* dcol, float* dimg, int B, int S, void* stream);
int sg2_nhwc_to_nchw_f32(const void* in, float* out, int B, int HW, int C, void* stream);
int sg2_nchw_f32_to_nhwc(const float* in, void* out, int B, int HW, int C, void* stream);

/* ---- small fp32 operators ---------------------------------------------------------------------------------
 * nn.Linear with M = batch rows (model.py:179, 217); x = cat(x1[M][K1], x2[M][K2]) (x2 may be NULL, K2 = 0). */
int sg2_linear_fwd(const float* x1, int K1, const float* x2, int K2, const float* w, const float* bias, void* out,
                   int out_bf16, int M, int N, void* stream);
int sg2_linear_bwd_w(const void* dy, int dy_bf16, const float* x1, int K1, const float* x2, int K2, float* dw,
                     float* dbias, int M, int N, int accumulate, void* stream);
/* dx = dy . w[:, :Kout]: two deterministic passes (per-slab partials in `scratch`, then their sum). */
int sg2_linear_bwd_x_scratch_floats(int N, int Kout);
int sg2_linear_bwd_x(const void* dy, int dy_bf16, const float* w, float* dx /* [M][Kout], overwritten */,
                     float* scratch /* sg2_linear_bwd_x_scratch_floats(N, Kout) floats */, int M, int N, int K, int Kout,
                     void* stream);
/* CA_NET GLU + reparameterisation (model.py:183-195): fc [B][4E] -> mu, logvar, c = eps*exp(.5 logvar)+mu */
int sg2_ca_glu_reparam_fwd(const float* fc, const float* eps, float* mu, float* logvar, float* c, int B, int E,
                           void* stream);
int sg2_ca_glu_reparam_bwd(const float* fc, const float* eps, const float* dmu, const float* dlogvar, const float* dc,
                           float* dfc, int B, int E, void* stream);
int sg2_chw_hwc_bf16(const void* in, void* out, int B, int C, int HW, int to_hwc, void* stream);
/* D logits: conv k4 s4 C->1 + bias + sigmoid on a 4x4 map (model.py:414-422) */
int sg2_logits_fwd(const void* x, const float* w, const float* bias, float* prob, int B, int HW, int C, void* stream);
int sg2_logits_bwd_scratch_floats(int B, int HW, int C);
int sg2_logits_bwd(const float* dprob, const float* prob, const void* x, const float* w, void* dx, int dx_accumulate,
                   float* dw /* += */, float* dbias /* += */,
                   float* dw_scratch /* sg2_logits_bwd_scratch_floats() floats when dw != NULL: per-sample-chunk partials */,
                   int B, int HW, int C, void* stream);
/* ---- losses (trainer.py:54-58, 298-311, 394-409, 439-446, 499) ---------------------------------------------
 * loss is a device scalar that the kernels ADD to (zero it first). probs/dprobs are contiguous [nvec][B]. */
int sg2_gan_bce(const float* probs, const float* targets, const float* weights, int nvec, int B, float* loss,
                float* dprobs, void* stream);
int sg2_kl_loss(const float* mu, const float* logvar, int n, float coeff, float* loss, float* dmu, float* dlogvar,
                void* stream);
int sg2_cal_loss(const float* x, const int* labels, int B, int F, float* ws, float* loss, float* dx, void* stream);
/* Adam (torch.optim.Adam semantics, betas from trainer.py:236-252) over a flat fp32 parameter bucket, fused with the
 * generator EMA (trainer.py:571-572; avg may be NULL). sg2_adam_tick increments the device-side step counter and
 * writes bc = {1 - beta1^t, sqrt(1 - beta2^t)} (device-resident so CUDA-graph replays stay correct). */
int sg2_adam_tick(int* step, float* bc, float beta1, float beta2, void* stream);
int sg2_adam_ema(float* p, const float* g, float* m, float* v, float* avg, long long n, float lr, float beta1,
                 float beta2, float eps, const float* bc, float ema_decay, void* p_bf16 /* optional bf16 mirror of p */,
                 void* stream);

/* ---- fp32-accurate ("precise") mode: relative error <= 1e-4 against the fp32 reference (model.py:125-128 runs fp32
 * end to end) ---------------------------------------------------------------------------------------------------
 * Activations and gradients are NHWC fp32. A convolution is SIX launches of sg2_conv_fprop / _dgrad / _wgrad on the
 * tcgen05 kernels above: sg2_split3 writes the three bf16 planes x = hi + mid + lo of an fp32 tensor (and of the fp32
 * weight packs from sg2_pack_weights_f32), and the cross terms (hi,hi) (hi,mid) (mid,hi) (hi,lo) (lo,hi) (mid,mid)
 * accumulate into one fp32 output (SG2_OUT_F32_ATOMIC without split-K adds each launch's tile exactly once). The
 * kernels below are the fp32 counterparts of the bandwidth-bound kernels; same arguments, float instead of bf16. */
int sg2_split3(const float* x, void* out /* bf16 [3][n] */, long long n, void* stream);
int sg2_pack_weights_f32(int kind, const float* w, float* wpk, float* wpkT, int Cout, int Cin, int Cout_pad, int Cin_pad,
                         int src_ohwi, void* stream);
int sg2_bn_stats_f32(const float* x, long long P, int C, int groups, double* stats, void* stream);
int sg2_bn_act_fwd_f32(const float* x, const double* stats, float* mean, float* rstd, const float* gamma,
                       const float* beta, const float* residual, float* out, long long P, int C, int groups, int act,
                       float eps, float momentum, float* running_mean, float* running_var,
                       long long* num_batches_tracked, void* stream);
int sg2_bn_act_bwd_f32(const float* x, const float* dout, const float* mean, const float* rstd, const float* gamma,
                       const float* beta, double* sums, float* dx, float* dgamma, float* dbeta, int accumulate,
                       long long P, int C, int groups, int act, void* stream);
/* mode 0: out = a + b;  mode 1: out = a > 0 ? b : 0.2 b (LeakyReLU backward, a = the activation's output) */
int sg2_ew_f32(int mode, const float* a, const float* b, float* out, long long n, void* stream);
/* in place on an fp32 conv output [B][H][W][C]: += bias9 (see sg2_conv_fprop; may be NULL), then act (0 | SG2_ACT_LRELU) */
int sg2_conv_post_f32(float* y, const float* bias9, int act, int B, int H, int W, int C, void* stream);
int sg2_concat_c_f32(const float* c, const float* h, float* out, int B, int HW, int E, int Ch, void* stream);
int sg2_concat_c_bwd_f32(const float* dcat, float* dh, float* dc /* += */, int B, int HW, int E, int Ch, void* stream);
int sg2_head_tanh_fwd_f32(const float* y, float* img, int B, int HW, int CP, void* stream);
int sg2_head_tanh_bwd_f32(const float* dimg, const float* img, float* dy, int B, int HW, int CP, void* stream);
int sg2_stem_im2col_f32(const float* img, float* col, int B, int S, void* stream);
int sg2_stem_col2im_f32(const float* dcol, float* dimg, int B, int S, void* stream);
int sg2_hwc_chw_f32(const float* in, float* out, int B, int HW, int C, int to_chw, void* stream);
int sg2_logits_fwd_f32(const float* x, const float* w, const float* bias, float* prob, int B, int HW, int C, void* stream);
int sg2_logits_bwd_f32(const float* dprob, const float* prob, const float* x, const float* w, float* dx,
                       int dx_accumulate, float* dw /* += */, float* dbias /* += */, int B, int HW, int C, void* stream);

#ifdef __cplusplus
}
#endif
#endif
