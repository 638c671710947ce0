/* fmri_b200.h — C ABI of libfmri_b200.so: the sm_100a kernels behind the VAE/GAN / WAE/GAN training step of
 * MariaPdg/thesis-fmri-reconstruction (models/vae_gan.py + the update logic of train/train_{vgan,wae}_stage*.py).
 *
 * The reference has no FFI of its own: every op below is reached in the reference through torch.nn / ATen.
 * Each entry point cites the reference call site whose arithmetic it replaces (paths relative to /root/reference).
 *
 * Conventions
 *  - extern "C"; plain pointers and sizes; no torch types.
 *  - return 0 on success, a negative fmri_status on error; fmri_last_error() gives a thread-local message.
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no call allocates device memory,
 *    synchronises the device, or touches host memory after returning. Workspaces are caller-owned.
 *  - activations are channels-last ("NHWC", [N,H,W,C] dense) in `dtype` (FMRI_BF16 -> tcgen05/TMEM/TMA tensor path,
 *    FMRI_F32 -> exact CUDA-core path). Master weights, gradients of weights, statistics and losses are fp32
 *    (statistic accumulators fp64). Weight tensors keep the reference layouts
 *    (Conv2d [Cout,Cin,5,5], ConvTranspose2d [Cin,Cout,5,5], Linear [out,in]).
 *  - all convolutions are 5x5, padding 2 (configs/models_config.py:3-5).
 */
#ifndef FMRI_B200_H
#define FMRI_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define FMRI_ABI_VERSION 8

typedef enum { FMRI_OK = 0, FMRI_ERR_ARG = -1, FMRI_ERR_UNSUPPORTED = -2, FMRI_ERR_CUDA = -3, FMRI_ERR_WORKSPACE = -4 } fmri_status;
typedef enum { FMRI_F32 = 0, FMRI_BF16 = 1 } fmri_dtype;
typedef enum { FMRI_ACT_NONE = 0, FMRI_ACT_RELU = 1, FMRI_ACT_TANH = 2, FMRI_ACT_SIGMOID = 3 } fmri_act;

int fmri_version(void);
const char* fmri_last_error(void);
/* number of kernels this library has launched since the last reset (memsets excluded) */
long long fmri_launch_count(int reset);
/* 1 when the running device is sm_100 and the tensor path can be used, 0 otherwise (no GPU: 0, no error). */
int fmri_tensor_path_available(void);

/* ---------------------------------------------------------------------------------------------------------
 * 5x5 convolutions on C>=32 channels — tcgen05 implicit GEMM (bf16) or direct CUDA-core conv (fp32).
 * Geometry is that of the FORWARD op: input [N,H,W,Cin] -> output [N,OH,OW,Cout],
 *   Conv2d:          OH = (H-1)/stride + 1                      (vae_gan.py:18-20, :118, :145)
 *   ConvTranspose2d: OH = 2H-1+output_pad, stride 2             (vae_gan.py:46-53)
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    int N, H, W, Cin, Cout;
    int stride;      /* 1 or 2 */
    int transposed;  /* 0 Conv2d, 1 ConvTranspose2d */
    int output_pad;  /* ConvTranspose2d only */
    int dtype;       /* fmri_dtype of activations and activation gradients */
} fmri_conv_desc;

void fmri_conv_out_hw(const fmri_conv_desc* d, int* OH, int* OW);
/* bf16 weight packs consumed by the tensor path: pack_f (fprop), pack_d (dgrad); the layout is private to the library
 * (tap-major [25][N][K], plus a parity-merged pack for layers with a 32-channel side). Each buffer holds
 * fmri_conv_pack_elems(d) bf16 elements. Refreshed after every optimizer step. Either pointer may be NULL. */
size_t fmri_conv_pack_elems(const fmri_conv_desc* d);
int fmri_conv_pack_weights(const fmri_conv_desc* d, const float* w, void* pack_f, void* pack_d, void* stream);
/* y = act(conv(x, w) + bias); optionally accumulates per-output-channel sum / sum-of-squares of the stored y into
 * fp64 stat_sum/stat_sq[Cout] (BatchNorm batch statistics, vae_gan.py:21). `w` fp32 master weights (used by the fp32
 * path), `pack_f` bf16 pack (used by the bf16 path). */
int fmri_conv_fprop(const fmri_conv_desc* d, const void* x, const float* w, const void* pack_f, const float* bias,
                    int act, void* y, double* stat_sum, double* stat_sq, void* stream);
/* Optional fusion for fmri_conv_dgrad: when dx is the upstream gradient of a bias+ReLU layer WITHOUT BatchNorm
 * (Discriminator.conv[0], vae_gan.py:145-147), `y` is that layer's post-ReLU output (same [N,H,W,Cin] layout and dtype as dx)
 * and the call applies its ReLU backward, dx *= (y > 0), in the data-gradient epilogue (saves the separate read-dy /
 * write-dx pass of fmri_relu_backward). */
typedef struct {
    const void* y;
    const unsigned* bits; /* optional: fmri_relu_bitmask() of `y` (32-channel tensors): the epilogue then reads 4 bytes per
                           * pixel instead of 64 */
} fmri_relu_mask;
/* dx = conv data-gradient of dy (replaces aten::convolution_backward input-grad); relu_mask nullable */
int fmri_conv_dgrad(const fmri_conv_desc* d, const void* dy, const float* w, const void* pack_d, void* dx,
                    const fmri_relu_mask* relu_mask, void* stream);
/* dw (+)= conv weight-gradient, reference layout fp32. Workspace: fmri_conv_wgrad_workspace() bytes. */
size_t fmri_conv_wgrad_workspace(const fmri_conv_desc* d);
int fmri_conv_wgrad(const fmri_conv_desc* d, const void* x, const void* dy, float* dw, int accumulate, void* ws,
                    size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Edge convolutions with a 3-channel image side kept in the module-boundary format (NCHW fp32):
 *   "in"  : Conv2d(3, C)  image -> C-channel NHWC activation   (Encoder.conv[0] vae_gan.py:74, Discriminator.conv[0] :145)
 *   "out" : Conv2d(C, 3)  C-channel NHWC activation -> image   (Decoder.conv[3] vae_gan.py:118-121, +bias +tanh)
 * C in {32, 64}. Up to three image sources are read back-to-back on the batch axis (the discriminator's torch.cat,
 * vae_gan.py:165) — pass the same pointer / NULL for unused ones and n_per_src = N for a single source.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    int N, H, W;  /* image-side grid for "in" (input image), C-side grid equals image grid for "out" (stride 1) */
    int C;        /* channel count of the wide side */
    int stride;   /* "in" only: 1 or 2 */
    int dtype;    /* dtype of the C-channel activation */
} fmri_edge_desc;
int fmri_edge_in_fprop(const fmri_edge_desc* d, const float* img0, const float* img1, const float* img2, int n_per_src,
                       const float* w, const float* bias, int act, void* y, void* ws, size_t ws_bytes, void* stream);
/* dimg[N,3,H,W] = data gradient wrt the concatenated image batch */
int fmri_edge_in_dgrad(const fmri_edge_desc* d, const void* dy, const float* w, float* dimg, void* ws, size_t ws_bytes,
                       void* stream);
/* dbias (nullable): also emits the bias gradient dbias[c] (+)= sum over pixels of dy (Discriminator.conv[0] has a bias) */
int fmri_edge_in_wgrad(const fmri_edge_desc* d, const float* img0, const float* img1, const float* img2, int n_per_src,
                       const void* dy, float* dw, float* dbias, int accumulate, void* ws, size_t ws_bytes, void* stream);
int fmri_edge_out_fprop(const fmri_edge_desc* d, const void* x, const float* w, const float* bias, int act, float* img,
                        void* ws, size_t ws_bytes, void* stream);
int fmri_edge_out_dgrad(const fmri_edge_desc* d, const float* dimg, const float* w, void* dx, void* ws, size_t ws_bytes,
                        void* stream);
int fmri_edge_out_wgrad(const fmri_edge_desc* d, const void* x, const float* dimg, float* dw, int accumulate, void* ws,
                        size_t ws_bytes, void* stream);
size_t fmri_edge_workspace(const fmri_edge_desc* d); /* 75*C floats, enough for every edge call */

/* ---------------------------------------------------------------------------------------------------------
 * Linear layers (nn.Linear: vae_gan.py:79,84-85,107,156,160,199,206-207,510-519)
 *   fprop: y[M,N] = act(x[M,K] w[N,K]^T + bias)      dgrad: dx[M,K] = dy[M,N] w[N,K]      wgrad: dw[N,K] (+)= dy^T x
 * Row pitches (elements) are explicit so K can be padded to the 16-byte TMA pitch (K = 3620 fMRI voxels -> 3624).
 * bf16 path operands: x / dy bf16; `wp` = bf16 copy of w with pitch ldw (fprop), `wpt` = bf16 copy of w^T [K,N]
 * with pitch ldwt (dgrad). fp32 path: x / dy fp32 and the fp32 master `w` (pitch K) is used directly.
 * y_dtype may be FMRI_F32 even on the bf16 path (latent heads, split-K accumulation).
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    int M, N, K;
    int dtype;
} fmri_linear_desc;
/* Padding columns (ldw > K, ldwt > N) are never written: zero-initialise a padded buffer once. Several layers may
 * share one pitched buffer (the l_mu / l_var heads are packed side by side, vae_gan.py:84-85). */
int fmri_linear_pack_weights(const fmri_linear_desc* d, const float* w, void* wp, int ldw, void* wpt, int ldwt,
                             void* stream);
int fmri_linear_fprop(const fmri_linear_desc* d, const void* x, int ldx, const float* w, const void* wp, int ldw,
                      const float* bias, int act, void* y, int ldy, int y_dtype, void* stream);
int fmri_linear_dgrad(const fmri_linear_desc* d, const void* dy, int lddy, const float* w, const void* wpt, int ldwt,
                      void* dx, int lddx, int dx_dtype, int accumulate /* fp32 dx only */, void* stream);
int fmri_linear_wgrad(const fmri_linear_desc* d, const void* x, int ldx, const void* dy, int lddy, float* dw,
                      int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * BatchNorm (train: batch statistics; momentum semantics of torch, momentum=0.9 in the reference) + ReLU on a
 * channels-last [rows, C] matrix. vae_gan.py:21,27-34,54,58-59,80-82,108-109,158-159,200-201
 * --------------------------------------------------------------------------------------------------------- */
int fmri_colstats(const void* x, int dtype, long long rows, int C, double* sum, double* sq, void* stream);
int fmri_bn_finalize(const double* sum, const double* sq, long long rows, int C, float eps, float momentum, float* mean,
                     float* invstd, float* running_mean, float* running_var, void* stream);
int fmri_bn_apply(const void* x, int x_dtype, void* y, int y_dtype, long long rows, int C, const float* mean,
                  const float* invstd, const float* gamma, const float* beta, int relu, void* stream);
/* dx, dgamma (+)=, dbeta (+)= ; train=0 treats mean/invstd as constants (eval-mode BN). ws: 3*C doubles. */
int fmri_bn_backward(const void* x, int x_dtype, const void* dy, void* dx, int g_dtype, long long rows, int C,
                     const float* mean, const float* invstd, const float* gamma, const float* beta, int relu, int train,
                     float* dgamma, float* dbeta, int accumulate, double* ws, void* stream);
/* The same with dx produced for rows [row0, row0 + nrows) only (dx points at the first of them): train-mode BatchNorm couples
 * all rows through the two sums, so those always run over the whole [rows, C] matrix, but a caller that needs the input
 * gradient of a few samples only (the discriminator's feature-tap sweep feeds ONE of its three image sources,
 * train_vgan_stage1.py:330-372 via vae_gan.py:163-175) skips the apply pass on the rest. */
int fmri_bn_backward_slice(const void* x, int x_dtype, const void* dy, void* dx, int g_dtype, long long rows, long long row0,
                           long long nrows, int C, const float* mean, const float* invstd, const float* gamma,
                           const float* beta, int relu, int train, float* dgamma, float* dbeta, int accumulate, double* ws,
                           void* stream);
/* Two upstreams a, b through one BatchNorm layer (two backward sweeps over the same saved forward state): the sums read x once
 * for both (3 passes instead of 4), the apply reads x once and writes both gradients (5 passes instead of 6). Each upstream's
 * dx equals that of fmri_bn_backward bit for bit (same kernels' arithmetic and row partition; only the order of the fp64
 * atomics behind the means may differ). dgamma / dbeta (nullable) take upstream a's parameter gradient. ws: 6*C doubles. */
int fmri_bn_backward_pair(const void* x, int x_dtype, const void* dy_a, const void* dy_b, void* dx_a, void* dx_b, int g_dtype,
                          long long rows, int C, const float* mean, const float* invstd, const float* gamma,
                          const float* beta, int relu, int train, float* dgamma, float* dbeta, int accumulate, double* ws,
                          void* stream);
/* The same with upstream b's dx produced for rows [row0, row0 + nrows) only (dx_b points at the first of them); dx_a covers
 * all rows and the sums of both run over all rows (the discriminator's class path and feature-tap sweeps through block 1). */
int fmri_bn_backward_pair_slice(const void* x, int x_dtype, const void* dy_a, const void* dy_b, void* dx_a, void* dx_b,
                                int g_dtype, long long rows, long long row0, long long nrows, int C, const float* mean,
                                const float* invstd, const float* gamma, const float* beta, int relu, int train,
                                float* dgamma, float* dbeta, int accumulate, double* ws, void* stream);
/* bits[pixel] bit j = (y[pixel][j] > 0): ReLU mask of a channels-last bf16 tensor with exactly 32 channels, 4 B per pixel
 * (consumed by fmri_conv_dgrad through fmri_relu_mask.bits) */
int fmri_relu_bitmask(const void* y, int dtype, long long pixels, int C, unsigned* bits, void* stream);
int fmri_relu_backward(const void* y, const void* dy, void* dx, int dtype, long long n, void* stream);
int fmri_colsum(const void* x, int dtype, long long rows, int C, float* out /* += */, void* stream);

/* layout / dtype converters: NCHW <-> NHWC (any of f32/bf16 on either side; flatten order of vae_gan.py:89,127,180),
 * and a 2-D cast with row pitch */
int fmri_nchw_to_nhwc(const void* src, int src_dtype, void* dst, int dst_dtype, int N, int C, int H, int W,
                      void* stream);
int fmri_nhwc_to_nchw(const void* src, int src_dtype, void* dst, int dst_dtype, int N, int C, int H, int W,
                      int accumulate, void* stream);
int fmri_cast2d(const void* src, int src_dtype, int lds, void* dst, int dst_dtype, int ldd, long long rows, int cols,
                void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Losses. vae_gan.py:266-269 (reparameterize), :302-320 (VaeGan.loss), train_wae_stage1.py:281-282,301-303
 * --------------------------------------------------------------------------------------------------------- */
/* mu / logvar have row pitch `ld` floats (the two halves of one [B, 2Z] head output); z, eps, kl dense. */
int fmri_reparam_kl_fwd(const float* mu, const float* logvar, int ld, const float* eps, float* z /*nullable*/,
                        float* kl /*nullable*/, int B, int Z, void* stream);
/* dmu / dlogvar (d_dtype, row pitch ldd) from gz = dL/dz (nullable) and dL/dkl = gkl[b] (or the constant gkl_const
 * when gkl is NULL: the reference sums kl over the batch, train_vgan_stage1.py:369). */
int fmri_reparam_kl_bwd(const float* mu, const float* logvar, int ld, const float* eps, const float* gz /*nullable*/,
                        const float* gkl /*nullable*/, float gkl_const, void* dmu, void* dlogvar, int ldd, int d_dtype,
                        int B, int Z, void* stream);
/* out[b] = scale * sum_j (a[b,j]-b[b,j])^2   (feature-matching MSE scale=.5 over 16384 features; NLE / WAE recon) */
int fmri_rowsqdiff_fwd(const void* a, const void* b, int dtype, float* out, long long rows, long long F, float scale,
                       void* stream);
int fmri_rowsqdiff_bwd(const void* a, const void* b, int dtype, const float* g, void* da, void* db, long long rows,
                       long long F, float scale, void* stream);
/* p = sigmoid(x w + b) for Linear(F,1)+sigmoid heads (vae_gan.py:160,183 / :519-520) */
int fmri_head_sigmoid_fwd(const void* x, int dtype, const float* w, const float* bias, float* p, int rows, int F,
                          void* stream);
int fmri_head_sigmoid_bwd(const void* x, int dtype, const float* w, const float* p, const float* gp, void* dx,
                          float* dw /* += */, float* db /* += */, int rows, int F, void* stream);
/* bce[i] = -scale*log(p+1e-3) (positive) or -scale*log(1-p+1e-3) */
int fmri_bce_fwd(const float* p, float* out, int n, int positive, float scale, void* stream);
int fmri_bce_bwd(const float* p, const float* g, float* dp, int n, int positive, float scale, int accumulate,
                 void* stream);
/* WAE-MMD latent penalty, inverse-multiquadratic kernel summed over the scales {.1,.2,.5,1,2,5,10} * 2 Z sigma2
 * (Tolstikhin et al.; the estimator of the repositories the reference's README.md:287,293 cites). EXTENSION: the
 * reference ships no MMD code (SURVEY.md 0-3), so this pair is pinned only against oracle/mmd.py ("parity unpinned").
 * zq = encoded latents [B, Z] (row pitch ldq floats, e.g. the mu half of a [B, 2Z] head output), zp = prior samples.
 *   fwd: mmd[0] = lambda * { [sum_{i!=j} k(q_i,q_j) + sum_{i!=j} k(p_i,p_j)] / (B(B-1)) - 2/B^2 sum_{i,j} k(q_i,p_j) }
 *        ws = 3 doubles of caller-owned scratch (zeroed by the call).
 *   bwd: dzq (+)= lambda * d mmd / d zq   (fp32, row pitch ldd floats). 2 <= B, Z <= 512. */
int fmri_mmd_imq_fwd(const float* zq, int ldq, const float* zp, int ldp, int B, int Z, float sigma2, float lambda,
                     float* mmd, double* ws, void* stream);
int fmri_mmd_imq_bwd(const float* zq, int ldq, const float* zp, int ldp, int B, int Z, float sigma2, float lambda,
                     float* dzq, int ldd, int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused multi-tensor optimizers over fp32 master weights (one launch per parameter bucket).
 * train_vgan_stage1.py:275-283 (RMSprop alpha=.9 eps=1e-8), train_wae_stage1.py:221-224 (Adam betas=(.5,.999)),
 * clamp>0 folds the `p.grad.data.clamp_(-1,1)` of train_vgan_stage2.py:391,406.
 * --------------------------------------------------------------------------------------------------------- */
/* lr_dev (nullable) overrides lr from device memory; gate_dev (nullable): the update is skipped when *gate_dev == 0
 * (the equilibrium gate of train_vgan_stage1.py:396-404 decided on the device by fmri_vgan_gate). */
int fmri_multi_tensor_rmsprop(int n, float* const* p, const float* const* g, float* const* sq, const int64_t* numel,
                              float lr, float alpha, float eps, float clamp, const float* lr_dev,
                              const float* gate_dev, void* stream);
int fmri_multi_tensor_adam(int n, float* const* p, const float* const* g, float* const* m, float* const* v,
                           const int64_t* numel, float lr, float beta1, float beta2, float eps, int step, float clamp,
                           const float* lr_dev, const float* gate_dev, void* stream);
/* The same with Adam's step count read from device memory (bias corrections 1 - beta^t computed on the device), and the kernel
 * that advances it: a training step with no host-side scalar that changes from step to step can be captured in a CUDA graph. */
int fmri_multi_tensor_adam_dev(int n, float* const* p, const float* const* g, float* const* m, float* const* v,
                               const int64_t* numel, float lr, float beta1, float beta2, float eps, const int* step_dev,
                               float clamp, const float* lr_dev, const float* gate_dev, void* stream);
int fmri_step_increment(int* step_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Glue of the fused training step (no reference counterpart as separate ops: autograd does these implicitly)
 * --------------------------------------------------------------------------------------------------------- */
/* out = (a*x + b*y) * (img ? 1 - img^2 : 1): mixes two image gradients (loss_decoder = lambda*mse - (1-lambda)*loss_dis,
 * train_vgan_stage1.py:372) and applies the tanh backward of Decoder.conv[3] (vae_gan.py:120). y, img nullable. */
int fmri_axpby_tanh_bwd(float a, const float* x, float b, const float* y, const float* img, float* out, long long n,
                        void* stream);
/* out[c] (+)= sum over n, hw of x[n,c,hw]  (bias gradient of Decoder.conv[3], NCHW fp32) */
int fmri_chansum_nchw(const float* x, int N, int C, long long HW, float* out, int accumulate, void* stream);
/* out[0] (+)= scale * sum x[0..n)  (the torch.sum of per-sample losses, train_vgan_stage1.py:369-372) */
int fmri_vecsum(const float* x, long long n, float scale, float* out, int accumulate, void* stream);
/* gates[0] = train_dis, gates[1] = train_dec (0.f / 1.f) from sums[0] = sum bce_original, sums[1] = sum bce_predicted
 * over `count` samples (train_vgan_stage1.py:396-404) */
int fmri_vgan_gate(const float* sums, float count, float margin, float equilibrium, float* gates, void* stream);
/* The same gate with the pre-gate value of train_dis as an argument: the loss-mix block of train_vgan_stage1.py:359-388
 * sets train_dis = False in mode 'vae' (:387) before the gate runs, and the gate's "neither -> both" rule (:403-404) can
 * turn it back on. fmri_vgan_gate is this call with train_dis_in = 1. */
int fmri_vgan_gate_mix(const float* sums, float count, float margin, float equilibrium, int train_dis_in, float* gates,
                       void* stream);
/* x[i] *= s for i < n (fp32, in place). Mode 'vae' (train_vgan_stage1.py:382-387) takes g_dec = lambda_mse * the decoder
 * weight gradients of d sum(nle) / d decoder, whose data gradient is the encoder's upstream at unit weight. */
int fmri_scale_f32(float* x, long long n, float s, void* stream);
/* eval-mode BatchNorm statistics: mean = running_mean, invstd = rsqrt(running_var + eps) */
int fmri_bn_eval_stats(const float* running_mean, const float* running_var, int C, float eps, float* mean,
                       float* invstd, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Inference side (SURVEY.md 8f-2) and the step's input edge (8f-3).
 * fmri_bn_fold: eval-mode BatchNorm folded into the preceding bias-free layer, w_out = w * gamma / sqrt(running_var + eps)
 *   per OUTPUT channel ((i / inner) % C: Conv2d inner = Cin*25, ConvTranspose2d inner = 25, Linear inner = in_features),
 *   b_out = beta - running_mean * that scale; the folded layer then runs conv / linear + bias + ReLU in ONE kernel
 *   (VaeGan.forward eval branch, vae_gan.py:288-297; inference/inference_gan.py:340-442).
 * fmri_pearson / fmri_ssim: PearsonCorrelation / StructuralSimilarity of train/train_utils.py:267-293, 295-425 on two
 *   fp32 NCHW batches (scalar results on the device; ws: 5 / 1 doubles).
 * fmri_image_pipeline: uint8 NHWC batch (1 or 3 channels) -> normalised fp32 NCHW: /255, GreyToColor, per-image horizontal
 *   flip (flip[n] != 0), per-image integer shift with edge replication (shift_yx[2n], [2n+1]), (v - mean) / std
 *   (train_vgan_stage1.py:161-171; data_preprocessing/data_loader.py:93-111, 187-217, 374-400). mean3 / std3 are HOST arrays.
 * --------------------------------------------------------------------------------------------------------- */
int fmri_bn_fold(const float* w, long long n, long long inner, int C, const float* running_mean, const float* running_var,
                 const float* gamma, const float* beta, float eps, float* w_out, float* b_out, void* stream);
int fmri_pearson(const float* a, const float* b, long long n, float* out, double* ws, void* stream);
int fmri_ssim(const float* a, const float* b, int N, int C, int H, int W, float* out, double* ws, void* stream);
int fmri_image_pipeline(const unsigned char* src, int N, int H, int W, int Csrc, const int* flip, const int* shift_yx,
                        const float* mean3, const float* std3, float* dst, void* stream);
/* fmri_image_rescale: the BOLD5000 stimulus transform Rescale -> RandomShift -> SampleToTensor -> Normalization
 *   (data_preprocessing/data_loader.py Rescale, :187-217 RandomShift, :93-111 Normalization; train/train_vgan_stage2.py:160-168)
 *   on native-resolution sources: N uint8 HWC images of any size and 1 or 3 channels, each described by one fmri_image_src
 *   (byte offset into `src`, which holds src_bytes bytes), -> normalised fp32 NCHW dst [N, 3, H, W]. Rescale is
 *   skimage.transform.resize(img, (H, W)) with its defaults (skimage >= 0.19: order 1, mode 'reflect', anti-aliasing when
 *   some axis downsamples, output in [0, 1]); per axis with f = in / out: a Gaussian pre-filter sigma = max(0, (f - 1) / 2),
 *   radius int(4 sigma + 0.5), mirror boundary, then linear interpolation at u = (o + 0.5) f - 0.5. Flip, shift, GreyToColor
 *   and normalisation are those of fmri_image_pipeline, applied to the resized image; with Hs = H and Ws = W the result is
 *   bit-identical to fmri_image_pipeline. fp32 weights and sums, no atomics: two calls give the same bits.
 *   `images` is a HOST array; every entry is checked before anything is launched (sizes >= 1 and <= 32768, C in {1, 3},
 *   the image inside src_bytes; FMRI_ERR_UNSUPPORTED when an image's source band does not fit the shared memory of one
 *   CTA), then the table is copied into ws (fmri_image_rescale_workspace(N) bytes, 8-byte aligned) on `stream`. ws must
 *   stay untouched until the kernel has run; nothing is read back from the device. Not capturable in a CUDA graph (the
 *   table is copied from host memory at call time). */
typedef struct {
    long long offset; /* byte offset of the image's first pixel in src */
    int H, W, C;      /* source height, width, channels (1 or 3); the image is dense HWC */
} fmri_image_src;
size_t fmri_image_rescale_workspace(int N); /* bytes; 0 for N < 1 */
int fmri_image_rescale(const unsigned char* src, size_t src_bytes, const fmri_image_src* images, int N, int H, int W,
                       const int* flip, const int* shift_yx, const float* mean3, const float* std3, float* dst, void* ws,
                       size_t ws_bytes, void* stream);
/* fmri_image_resample: the COCO Stage-I loader's PIL / torchvision resize (Resize, CenterCrop, RandomResizedCrop on PIL
 *   images: PIL.Image.resize with BILINEAR or BICUBIC; train/train_vgan_stage1.py:161-171, data_preprocessing/data_loader.py
 *   :346 CocoDataloader) -> RandomHorizontalFlip / shift -> ToTensor -> GreyToColor -> Normalize, on native-resolution
 *   uint8 sources. Image n is the window described by images[n]: H x W pixels of C (1 or 3) interleaved channels at byte
 *   offset `offset` of `src` (src_bytes bytes), rows `pitch` bytes apart, so a crop of a larger image is a strided window
 *   and, as with PIL's crop-then-resize, the filter taps are clamped at the window's edges. The window is resized to
 *   Hr x Wr exactly as Pillow's 8-bit Image.resize does (fp64 filter weights, 22-bit fixed-point taps, a horizontal
 *   then a vertical pass, each rounded and clamped to uint8), and the H x W (the call's H, W) part of it at (oy, ox) is
 *   kept, which is Resize followed by CenterCrop without computing the discarded pixels. Flip, shift, GreyToColor and
 *   normalisation are those of fmri_image_pipeline: dst [N, 3, H, W] is bit-identical to fmri_image_pipeline applied to
 *   Pillow's uint8 result, and with Hr = H = window height, Wr = W = window width to fmri_image_pipeline on the source.
 *   Integer sums, no atomics: two calls give the same bits. `filter` is FMRI_RESAMPLE_BILINEAR or FMRI_RESAMPLE_BICUBIC
 *   (Pillow's Image.Resampling values). The taps are computed on the device, per CTA.
 *   `images` is a HOST array; every entry is checked before anything is launched: sides >= 1 and <= 32768, C in {1, 3},
 *   pitch >= W * C, the window inside src_bytes, oy + H <= Hr and ox + W <= Wr. An image whose one-row band needs more
 *   than FMRI_RESAMPLE_MAX_SMEM bytes of shared memory is refused with FMRI_ERR_UNSUPPORTED, also before any launch. Per
 *   axis, with `in` the window side and `out` the resized side, Pillow's support is sup = s max(in / out, 1) (s = 1
 *   bilinear, 2 bicubic) and its tap count k = 2 ceil(sup) + 1. A band of `ty` output rows needs, each term rounded up to
 *   16 bytes: 4 W k_x + 8 W (horizontal taps) + 4 ty k_y + 8 ty (vertical taps) + rows W C (the uint8 horizontal-pass
 *   rows it reads), rows = min(window H, (int)((ty - 1) in_y / out_y + 2 sup_y) + 2); for a window more than 100 times
 *   taller than wide that shrinks vertically, which Image.resize (and this call) resamples vertically first, the last
 *   term is ty Wwin C instead. E.g. 480 x 640 -> 64 x 64 BICUBIC takes 17296 B at ty = 1; a window 4096 wide resized
 *   to 64 columns BICUBIC (k_x = 257) about 65 KB; 32768 -> 64 columns does not fit. The table is then copied into ws
 *   (fmri_image_resample_workspace(N) bytes, 8-byte aligned) on `stream`. ws must stay untouched until the kernel has
 *   run; nothing is read back from the device. Not capturable in a CUDA graph. */
#define FMRI_RESAMPLE_MAX_SMEM 232448 /* 227 KB: the opt-in shared memory of one CTA on sm_100 */
typedef enum { FMRI_RESAMPLE_BILINEAR = 2, FMRI_RESAMPLE_BICUBIC = 3 } fmri_resample_filter;
typedef struct {
    long long offset; /* byte offset of the window's top-left pixel in src */
    long long pitch;  /* bytes from one window row to the next (>= W * C) */
    int H, W, C;      /* window height, width, channels (1 or 3) */
    int Hr, Wr;       /* size of the whole resized image */
    int oy, ox;       /* top-left corner of the call's H x W output inside the Hr x Wr resized image */
} fmri_image_window;
size_t fmri_image_resample_workspace(int N); /* bytes; 0 for N < 1 */
int fmri_image_resample(const unsigned char* src, size_t src_bytes, const fmri_image_window* images, int N, int H, int W,
                        int filter, const int* flip, const int* shift_yx, const float* mean3, const float* std3, float* dst,
                        void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * All-pairs similarity and n-way identification: the exhaustive, exact-expectation form of the reference's sampled
 * objective_assessment (train/train_utils.py:752).
 * fmri_pairwise_similarity: out[i, j] (fp32, [N, M] row-major) = the metric of pred[i] (of [N, C, H, W]) against
 *   target[j] (of [M, C, H, W]), both fp32 NCHW:
 *     FMRI_METRIC_PCC  PearsonCorrelation()(pred[i:i+1], target[j:j+1])      (train_utils.py:267-293)
 *     FMRI_METRIC_SSIM StructuralSimilarity()(pred[i:i+1], target[j:j+1])    (train_utils.py:295-425; the window and
 *                      constants of fmri_ssim; H or W below 11 is FMRI_ERR_UNSUPPORTED)
 *   ws: fmri_pairwise_workspace() bytes, 16-byte aligned (FMRI_ERR_WORKSPACE when smaller). CUDA-core fp32 with fp64
 *   accumulation, no atomics: two calls on the same inputs give the same bits.
 * fmri_identification: from a square similarity matrix sim [N, N] (row i: reconstruction i, column i: its own target),
 *   wins[i] = #{j != i : sim[i, i] > sim[i, j]} (strict; NaN never wins) and, for each n = ns[q] (a HOST array,
 *   2 <= n <= N), acc[q] = (1/N) sum_i C(wins[i], n-1) / C(N-1, n-1): the probability that the true target beats n-1
 *   distractors drawn uniformly without replacement, averaged over the rows, in fp64.
 * Every argument is checked before the first launch (FMRI_ERR_ARG for N < 2, n outside [2, N], non-positive sizes).
 * --------------------------------------------------------------------------------------------------------- */
typedef enum { FMRI_METRIC_PCC = 0, FMRI_METRIC_SSIM = 1 } fmri_metric;
size_t fmri_pairwise_workspace(int N, int M, int C, int H, int W, int metric); /* bytes; 0 for invalid arguments */
int fmri_pairwise_similarity(const float* pred, int N, const float* target, int M, int C, int H, int W, int metric,
                             float* out, void* ws, size_t ws_bytes, void* stream);
int fmri_identification(const float* sim, int N, const int* ns, int n_count, int* wins, double* acc, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FMRI_B200_H */
