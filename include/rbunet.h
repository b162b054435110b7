/*
 * rbunet.h — C ABI of librbunet.so: the B200 (sm_100a) Robust U-Net hot path.
 *
 * The reference (UofgCoastline/EUSIPCO-2026-Robust-Unet) has no FFI: its hot path is the set of
 * PyTorch ops dispatched by `RobustUNet.forward` (Main_Final.py:290-321), `nn.BCELoss`
 * (Main_Final.py:551,580) and `ModelEvaluator.calculate_metrics` (Main_Final.py:519-547).
 * Each entry point below replaces the ATen/cuDNN dispatch of the reference lines it cites
 * (SURVEY.md §2.1 maps ATen ops to kernels).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *  - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *  - the caller allocates and frees every buffer (including workspaces); the library keeps no tensor state;
 *  - every function enqueues on `stream` (a cudaStream_t passed as void*) and returns immediately;
 *  - return value: 0 on success, negative on error (RBU_ERR_*); rbu_last_error() gives the message;
 *    nothing throws or exits across the ABI; unsupported input is an error, there is NO CPU fallback;
 *  - activations are NHWC bf16 "views": pointer to the first channel of a channel slice, pixel stride
 *    `ld` in elements (multiple of 8), `C` channels in the slice (multiple of 8);
 *  - "pixels" P = N*H*W.
 */
#ifndef RBUNET_H_
#define RBUNET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBU_OK 0
#define RBU_ERR_INVALID (-1)
#define RBU_ERR_CUDA (-2)
#define RBU_ERR_UNSUPPORTED (-3)

/* ------------------------------------------------------------------ library */
int rbu_version(void);
const char* rbu_last_error(void);
/* 0 if the current device is compute capability 10.x (tcgen05/TMEM/TMA available). */
int rbu_device_check(void);
int rbu_sm_count(void);
/* Number of CUDA kernels this library has launched in the calling process (bench.py's gpu_launches). */
unsigned long long rbu_launch_count(void);

/* ------------------------------------------------------------------ input preprocessing
 * uint8 RGB [B,H,W,3] -> fp32 NCHW [B,n_channels,H,W]: ToTensor + Normalize(ImageNet) of Main_Final.py:697-701 in
 * channels 0-2; n_channels 4 appends the HSV saturation plane, 6 appends H/360, S, V (OpenCV float semantics; the
 * reference has no HSV code, SURVEY.md §8c).  Bit-identical to the numpy oracle. */
int rbu_preprocess(const uint8_t* img, int B, int H, int W, int n_channels, float* out, void* stream);

/* ------------------------------------------------------------------ image operations either side of the network
 * (SURVEY.md 8(f) rows 3 and 4; integer / byte work, bit-exact against the reference's numpy / OpenCV code)
 *
 * rbu_enhance_image: tif_to_image.py:139-171 enhance_image (duplicated at train_water_segmentation.py:103-174 and
 * predict_coastline.py:545-581).  img: [B,H,W,C] interleaved unsigned samples of `bits` (8 or 16) bits, C <= 8 bands.
 * Per image and band: p2, p98 = np.percentile(band, [2, 98]) (linear method, float64), then
 * clip((x - p2) / (p98 - p2) * 255, 0, 255); with enhance_water band 0 is multiplied by 0.7 where the stretched value is
 * below 100; truncation to uint8.  out: [B,H,W,C] uint8.  percentiles_out: optional [B,C,2] float64 device buffer.
 * A constant band (p98 == p2) yields 0 where the reference's NaN -> integer conversion is undefined. */
size_t rbu_enhance_workspace_bytes(int B, int C, int bits);
int rbu_enhance_image(const void* img, int bits, int B, int H, int W, int C, int enhance_water, uint8_t* out,
                      double* percentiles_out, void* workspace, size_t workspace_bytes, void* stream);
/* rbu_coastline_mask: predict_coastline.py:595-602 -- cv2.dilate(mask, getStructuringElement(MORPH_ELLIPSE, (k,k)),
 * iterations=1) - mask on uint8 [B,H,W] masks (any values; uint8 arithmetic), 1 <= ksize <= 64.  Contour tracing
 * (cv2.findContours / approxPolyDP, :605-616) stays on the host. */
int rbu_coastline_mask(const uint8_t* mask, int B, int H, int W, int ksize, uint8_t* out, void* stream);
/* Resizing of uint8 images (C = 3, RGB) and masks (C = 1), bit-exact with the library calls of the reference.  One
 * launch per call for a batch of sources of different sizes, all resized to oh x ow.  srcs_device: DEVICE array of B
 * descriptors (row_pitch in bytes >= W*C; the C bytes of a pixel are contiguous).  max_h / max_w bound every source's
 * H / W and size the bilinear weight tables; a descriptor outside them is skipped (its output is left unwritten).
 * out: [B,oh,ow,C] uint8.
 *  mode 0  Pillow Image.resize(BILINEAR) = torchvision transforms.Resize on PIL images (Main_Final.py:697-701,
 *          predict_coastline.py:386-392): Pillow's antialiasing two-pass fixed-point filter.  Downscales needing more
 *          than RBU_RESIZE_MAX_TAPS taps per output (factor > 127) return RBU_ERR_UNSUPPORTED.
 *  mode 1  Pillow Image.resize(NEAREST): the mask resize of Main_Final.py:44-54.
 *  mode 2  cv2.resize(INTER_NEAREST): the predicted mask back to scene size (predict_coastline.py:583-602).
 * Pinned against Pillow 12.2, OpenCV 4.13 and torchvision 0.26. */
#define RBU_RESIZE_MAX_TAPS (255)
typedef struct { const uint8_t* src; long long row_pitch; int H, W; } rbu_resize_src;
int rbu_resize_u8(const rbu_resize_src* srcs_device, int B, int C, int max_h, int max_w, int oh, int ow, int mode,
                  uint8_t* out, void* stream);

/* ------------------------------------------------------------------ tensor-core implicit GEMM
 * Replaces aten::convolution for 3x3 (dilation 1/2/4), 1x1 and ConvTranspose2d(2, stride 2)
 * (Main_Final.py:157,159,172,126,131,205-208,261-270) and, with re-packed weights, their data
 * gradients.  D[pixel, n] = sum over segments, taps, channels of X[pixel + tap, c] * W[n, tap, c].
 */
typedef struct {
  const void* x;   /* bf16 NHWC view of the input (for gather: the 2H x 2W tensor)            */
  int64_t x_ld;    /* pixel stride in elements                                               */
  int C;           /* channels in the slice = per-tap K extent                               */
  const void* w;   /* bf16 packed weights [Ncols][taps][C]                                   */
  int taps;        /* 1 (1x1), 9 (3x3) or 4 (gather=1: 2x2 stride-2 gather, tap = 2*i + j)   */
  int dil;         /* dilation of the 3x3 taps (padding == dilation)                         */
  int gather;      /* 1: X[pixel(n,h,w), tap(i,j)] = x[n, 2h+i, 2w+j] (ConvTranspose dgrad)  */
} rbu_gemm_operand;

typedef struct {
  int N, H, W;              /* pixel grid of the GEMM M dimension                                  */
  int nseg;                 /* 1 or 2 accumulated segments (e.g. conv1 dgrad + shortcut dgrad)     */
  rbu_gemm_operand seg[2];
  int Ncols;                /* GEMM N (Cout, or 4*Cout when scatter=1); multiple of 8              */
  void* y;                  /* bf16 NHWC output view                                               */
  int64_t y_ld;
  int scatter;              /* 1: ConvTranspose2d pixel shuffle: column (2i+j)*Cout+co of pixel    */
  int Cout;                 /*    (n,h,w) goes to y[n, 2h+i, 2w+j, co]; y is [N,2H,2W]; else 0     */
  const float* bias;        /* fp32 [Cout] or NULL                                                 */
  const void* addend;       /* optional bf16 NHWC view added to the result (scatter=0 only)        */
  int64_t addend_ld;
  const float* scale;       /* optional fp32 [Cout]: y = scale*acc + bias (eval-mode BatchNorm folded into the conv) */
  int relu;                 /* ReLU after scale / bias / addend on output channels [0, relu) (0: none);        */
                            /* a multiple of 8 (the epilogue works on 8-channel groups), at most Ncols (Cout   */
                            /* when scatter=1); anything else is RBU_ERR_INVALID                               */
  float* stats;             /* optional: rbu_conv_stats_floats(Ncols) floats receiving one row per CTA of      */
                            /* partial sum / sum of squares per output column of the STORED (bf16) result --  */
                            /* the BatchNorm batch statistics, fused into the epilogue (scatter=0 only)        */
  float* tile_stats;        /* optional (3x3 dilation-1 convs on >= 16x16 images, Ncols % 32 == 0):            */
                            /* rbu_conv_tile_stats_floats() floats receiving, per image and 16x8-pixel          */
                            /* half-tile, the column sum / sum of squares / max / min of the STORED result:     */
                            /* [N][chunks][4][Ncols] with chunks = rbu_conv_tile_stats_chunks(H, W)             */
} rbu_conv_gemm_args;

int rbu_conv_gemm(const rbu_conv_gemm_args* args, void* stream);
size_t rbu_conv_stats_floats(int Ncols);
int rbu_conv_tile_stats_chunks(int H, int W);
size_t rbu_conv_tile_stats_floats(int N, int H, int W, int Ncols);
/* nn.BatchNorm2d train-mode affine (Main_Final.py:158,173,127,132,210) from the partials above: columns
 * [col_off, col_off + C) of a conv whose GEMM had Ncols columns, `count` = N*H*W values per channel.  Updates the
 * running statistics (momentum, unbiased variance) when running_mean != NULL. */
int rbu_bn_finalize_partials(const float* part, int Ncols, int col_off, int C, int64_t count, const float* gamma,
                             const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                             float* scale, float* shift, float* mean_out, float* rstd_out, void* stream);

/* Re-pack fp32 torch-layout weights into the bf16 GEMM operand [Nn][T][K] (K contiguous).
 *  mode 0: Conv2d weight [Nn=Cout][K=Cin][T] for the forward GEMM
 *  mode 1: Conv2d weight [K=Cout][Nn=Cin][T] for the data gradient (taps rotated by 180 degrees)
 *  mode 2: ConvTranspose2d weight [K=Cin][Cout][2][2] for the forward GEMM (Nn = 4*Cout, T = 1)
 *  mode 3: ConvTranspose2d weight [Nn=Cin][K=Cout][2][2] for the data gradient (T = 4)
 * Replaces nothing in the reference (layout change only; Main_Final.py:157-172,261-270 parameters). */
int rbu_pack_weight(const float* src, void* dst, int Nn, int T, int K, int mode, int Cout, void* stream);

/* Every weight operand of a model in one launch.  `jobs_device` is a DEVICE array of njobs descriptors sorted by
 * first_block (job i owns blocks [first_block_i, first_block_i + rbu_pack_job_blocks(Nn, T, K, mode)); total =
 * Nn*T*K destination elements).  mode 0-3 as rbu_pack_weight; mode 4 builds the stem operand [2C][Kp] from the 3x3
 * conv1 weight (src) and the 1x1 shortcut weight (src2): Nn = 2C, K = Kp, T = input channels. */
typedef struct {
  const float* src;
  const float* src2;
  void* dst;
  long long first_block;
  long long total;
  int Nn, T, K, mode, Cout, reserved;
} rbu_pack_job;
long long rbu_pack_job_blocks(int Nn, int T, int K, int mode);
int rbu_pack_weights_multi(const rbu_pack_job* jobs_device, int njobs, long long total_blocks, void* stream);

/* Fused multi-tensor Adam with coupled L2 weight decay = torch.optim.Adam(params, lr, betas, eps, weight_decay) as used
 * by the reference (Main_Final.py:552,582), one launch for all parameter tensors.  `jobs_device`: DEVICE array sorted by
 * first_block (1024 elements per block); step is the 1-based step count of the bias corrections.  Hyper-parameters are
 * doubles: torch evaluates 1-beta^t, lr/(1-beta1^t) and sqrt(1-beta2^t) in Python doubles and only then rounds to fp32. */
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  long long first_block;
  long long numel;
} rbu_adam_job;
int rbu_adam_step(const rbu_adam_job* jobs_device, int njobs, long long total_blocks, double lr, double beta1, double beta2,
                  double eps, double weight_decay, int step, void* stream);

/* TEST-ONLY device reference: direct (CUDA-core) convolution, bf16 NHWC in, fp32 torch-layout weights
 * (rounded to bf16 on the fly), fp32 dense NHWC out.  Used by the parity tests at sizes where the CPU
 * oracle is too slow; never called by the product path. */
int rbu_conv_direct_ref(const void* x, int64_t x_ld, int N, int H, int W, int Cin, const float* w,
                        const float* bias, int Cout, int ksz, int dil, float* out, void* stream);

/* ------------------------------------------------------------------ loss + metrics (K9)
 * rbu_loss_forward replaces nn.BCELoss()(outputs, masks) (Main_Final.py:551,580) and, in the same
 * pass, the per-image confusion counts behind ModelEvaluator.calculate_metrics (Main_Final.py:519-547).
 * loss = w_bce * BCE + w_dice * (1 - (2*sum(p*y)+smooth)/(sum(p)+sum(y)+smooth)); defaults (1,0) are
 * reference-exact.  probs/target: fp32 [B*HW]; counts: int64 [B][4] = TP,FP,FN,TN for p > threshold
 * (strict); sums_out: double[4] = sum(bce), sum(p), sum(y), sum(p*y) (kept for the backward). */
size_t rbu_loss_workspace_bytes(int B, int64_t HW);
int rbu_loss_forward(const float* probs, const float* target, int B, int64_t HW, float threshold, float w_bce,
                     float w_dice, float smooth, void* workspace, size_t workspace_bytes, float* loss_out,
                     double* sums_out, int64_t* counts, void* stream);
/* dL/dprobs with torch's binary_cross_entropy_backward formula ((p-y)/max(p(1-p),1e-12)/N), times
 * grad_out[0] (NULL = 1). */
int rbu_loss_backward(const float* probs, const float* target, int64_t total, const float* grad_out,
                      const double* sums, float w_bce, float w_dice, float smooth, float* dprobs, void* stream);
/* Integer TP/FP/FN/TN per image only (Main_Final.py:521-535). */
int rbu_confusion_counts(const float* pred, const float* target, int B, int64_t HW, float threshold,
                         int64_t* counts, void* stream);

/* ------------------------------------------------------------------ weight-gradient GEMM (K11)
 * out[(m*Cb + n)*taps + t] (+)= sum_pixels A[p, m] * B[p (+) tap t, n]   (fp32, torch parameter layout)
 *   Conv2d:            A = dy (Ca = Cout), B = x (Cb = Cin), taps 1|9, dilation dil -> weight.grad [Cout,Cin,kh,kw]
 *   ConvTranspose2d:   A = x  (Ca = Cin),  B = dout [N,2H,2W] gathered per quadrant (gather=1, taps=4)
 *                                                                          -> weight.grad [Cin,Cout,2,2]
 * Replaces aten::convolution_backward (weight) of Main_Final.py:157,159,172,126,131,205-208,261-270.
 * Split-K partials live in the caller's workspace; the reduction order is fixed (deterministic). */
typedef struct {
  int N, H, W;      /* pixel grid of A (gather: the low-resolution grid)           */
  const void* a;    /* bf16 NHWC view, M = Ca channels                             */
  int64_t a_ld;
  int Ca;
  const void* b;    /* bf16 NHWC view, N = Cb channels (gather: the [N,2H,2W] map) */
  int64_t b_ld;
  int Cb;
  int taps, dil, gather;
  float* out;
  int accumulate;   /* 1: add to out, 0: overwrite                                 */
} rbu_wgrad_args;
size_t rbu_wgrad_workspace_bytes(const rbu_wgrad_args* args);
int rbu_wgrad_gemm(const rbu_wgrad_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ forward block kernels (K2-K8)
 * BatchNorm2d statistics + affine (Main_Final.py:158,160,173,127,132,210): scale = gamma*rstd,
 * shift = beta - mean*scale; training=1 uses batch statistics (biased variance) and updates the running
 * buffers (momentum, unbiased variance); training=0 uses the running buffers.  pool=1 additionally emits
 * per-(n,c) mean/max/min over H*W of the raw input — the AdaptiveAvg/MaxPool2d of ChannelAttention
 * (Main_Final.py:87-88,98-99); the arg-max needed by the backward pass is found by rbu_sa_reduce.
 * All elementwise kernels below need C = a power of two in [8, 2048]. */
size_t rbu_bn_stats_workspace_bytes(int N, int HW, int C);
int rbu_bn_stats(const void* x, int64_t ld, int N, int HW, int C, int pool, int training, const float* gamma,
                 const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                 float* scale, float* shift, float* mean_out, float* rstd_out, float* nc_mean, float* nc_max,
                 float* nc_min, void* workspace, size_t workspace_bytes, void* stream);
/* y = [relu](scale[c]*x + shift[c]) * drop[n,c]   (BN apply + ReLU + Dropout2d; Main_Final.py:182-184,220-221) */
/* The same outputs as rbu_bn_stats from partials in the [N][chunks][4][C] layout (sum, sum of squares, max, min per
 * chunk) that the 3x3 convolution epilogue writes (rbu_conv_gemm_args.tile_stats; chunks =
 * rbu_conv_tile_stats_chunks(H, W)): no pass over the activation tensor.  workspace: N*2*C doubles. */
int rbu_bn_stats_from_partials(const float* partials, int chunks, int N, int HW, int C, int pool, int training,
                               const float* gamma, const float* beta, float* running_mean, float* running_var,
                               float momentum, float eps, float* scale, float* shift, float* mean_out, float* rstd_out,
                               float* nc_mean, float* nc_max, float* nc_min, void* workspace, size_t workspace_bytes,
                               void* stream);
int rbu_affine_act(const void* x, int64_t x_ld, void* y, int64_t y_ld, int64_t P, int HW, int C, const float* scale,
                   const float* shift, const float* drop, int relu, void* stream);
/* ChannelAttention gate (Main_Final.py:97-101) from the pooled statistics; also A2g = scale*g, B2g = shift*g,
 * tv[n,c] = the raw extreme the max-pool selected (max if scale >= 0 else min) and nc_arg[n,c] reset to INT_MAX. */
int rbu_ca_gate(const float* nc_mean, const float* nc_max, const float* nc_min, const float* scale,
                const float* shift, const float* V1, const float* V2, int N, int C, int Ch, float* g, float* A2g,
                float* B2g, float* u_avg, float* u_max, float* h_avg, float* h_max, float* tv, int* nc_arg,
                void* stream);
/* SpatialAttention (Main_Final.py:112-117): channel mean/max (+argmax) of A2g*y2+B2g, then the 7x7 gate.  The same
 * pass records nc_arg[n,c] = first pixel with y2 == tv[n,c] (the AdaptiveMaxPool2d arg-max for the backward).
 * amax_out == NULL (inference) skips both arg-max outputs; tv and nc_arg may then be NULL too. */
int rbu_sa_reduce(const void* y2, int64_t ld, int64_t P, int HW, int C, const float* A2g, const float* B2g,
                  const float* tv, int* nc_arg, float* s_out /* [P][2] */, int* amax_out, void* stream);
int rbu_sa_gate(const float* s, int N, int H, int W, const float* k7, float* gs, void* stream);
/* out = relu((A2g*y2+B2g)*gs + r), r = As*ys+Bs (projection) or the identity input (Main_Final.py:179,190-194) */
int rbu_rb_out(const void* y2, int64_t y2_ld, const void* rsrc, int64_t r_ld, void* out, int64_t out_ld, int64_t P,
               int HW, int C, const float* A2g, const float* B2g, const float* gs, const float* As, const float* Bs,
               void* stream);
/* nn.MaxPool2d(2) (Main_Final.py:235,239,243,249) */
int rbu_maxpool2x2(const void* x, int64_t x_ld, void* y, int64_t y_ld, int N, int Ho, int Wo, int C, void* stream);
/* AttentionGate (Main_Final.py:143-148): q0 = w_psi . relu(BN_g(yg) + BN_x(yx)) + b_psi, BatchNorm2d(1)
 * statistics -> stats[4] = {scale, shift, mean, rstd}; then out = skip * sigmoid(scale*q0 + shift). */
int rbu_ag_psi_blocks(int64_t P, int F);  /* partials needs 2*blocks floats */
int rbu_ag_psi(const void* yg, int64_t yg_ld, const void* yx, int64_t yx_ld, int64_t P, int F, const float* Ag,
               const float* Bg, const float* Ax, const float* Bx, const float* wpsi, const float* bpsi, int training,
               const float* gamma, const float* beta, float* running_mean, float* running_var, float momentum,
               float eps, float* q0, float* stats, float* partials, void* stream);
int rbu_ag_apply(const void* skip, int64_t s_ld, void* out, int64_t o_ld, int64_t P, int C, const float* q0,
                 const float* stats, float* psi, void* stream);
/* Stem: fp32 NCHW image -> bf16 3x3 patches [P][Kp] (k = tap*nc + c) so inc.conv1 + inc.shortcut
 * (Main_Final.py:157,172,233) run as one tensor-core GEMM. */
int rbu_stem_im2col(const float* x, int N, int nc, int H, int W, int Kp, void* out, void* stream);
/* outc (Main_Final.py:274-277,321): probs = sigmoid(w.x + b) in fp32; logits optional. */
int rbu_head_forward(const void* x, int64_t ld, int64_t P, int C, const float* w, const float* b, float* probs,
                     float* logits, void* stream);

/* ------------------------------------------------------------------ backward block kernels (K12)
 * Replace the autograd nodes of the same reference lines (native_batch_norm_backward, threshold_backward,
 * sigmoid_backward, mul/add/sum, adaptive_max_pool2d_backward, max_pool2d_with_indices_backward). */
size_t rbu_bwd_workspace_bytes(int N, int HW, int C);
int rbu_head_backward(const float* dprobs, const float* probs, const void* x, int64_t x_ld, void* dx, int64_t dx_ld,
                      int64_t P, int C, const float* w, float* dw, float* db, void* workspace, size_t workspace_bytes,
                      void* stream);
/* ResidualBlock backward in three passes over the activations (SURVEY.md Appendix C):
 *  rbu_rb_bwd1: de = dout*[out>0] (may alias dout); dG[p] = sum_c de*(A2g*y2+B2g); shortcut: sums_s_raw = sum de, sum de*ys
 *  rbu_sa_bwd : SpatialAttention backward on the per-pixel maps -> ds[P][2], dk7[98]
 *  rbu_rb_bwd2: D[N][2][C] (double) = per-(n,c) sum dc, sum dc*y2;  dc = de*gs + ds_avg/C + ds_max*[c == argmax_c]
 *  rbu_rb_mid : ChannelAttention MLP backward, BatchNorm sums (sums2 = dbeta2|dgamma2, sums_s likewise) and the
 *               coefficients of the last pass, all from D and forward statistics (no pass over the data)
 *  rbu_rb_bwd3: dy2 = c1*dc + c0 + cy*y2 + cm*[pixel == nc_arg]; dys = es*de + e0 + ey*ys */
int rbu_rb_bwd1(const void* dout, int64_t dout_ld, const void* out, int64_t out_ld, const void* y2, int64_t y2_ld,
                void* de, int64_t de_ld, const void* ys, int64_t ys_ld, int N, int HW, int C, const float* A2g,
                const float* B2g, float* dG, float* sums_s_raw, void* workspace, size_t workspace_bytes, void* stream);
int rbu_sa_bwd(const float* dG, const float* gs, const float* s, int N, int H, int W, const float* k7, float* ds,
               float* dk7, void* workspace, size_t workspace_bytes, void* stream);
int rbu_rb_bwd2(const void* de, int64_t de_ld, const void* y2, int64_t y2_ld, int N, int HW, int C, const float* gs,
                const float* ds, const int* amax_c, double* D, void* workspace, size_t workspace_bytes, void* stream);
int rbu_rb_mid(const double* D, const float* g, const float* h_avg, const float* h_max, const float* u_avg,
               const float* u_max, const float* nc_mean, const float* tv, const float* V1, const float* V2,
               const float* scale2, const float* shift2, const float* mean2, const float* rstd2, int N, int HW, int C,
               int Ch, float* scratch, float* dV1, float* dV2, float* sums2, float* coef, const float* sums_s_raw,
               const float* scale_s, const float* mean_s, const float* rstd_s, float* sums_s, float* coef_s, void* stream);
int rbu_rb_bwd3(const void* de, int64_t de_ld, const void* y2, int64_t y2_ld, void* dy2, int64_t dy2_ld, const void* ys,
                int64_t ys_ld, void* dys, int64_t dys_ld, int N, int HW, int C, const float* gs, const float* ds,
                const int* amax_c, const int* nc_arg, const float* coef, const float* coef_s, void* stream);
int rbu_bn_bwd(const void* dy, int64_t dy_ld, const void* y, int64_t y_ld, void* dx, int64_t dx_ld, int N, int HW,
               int C, const float* scale, const float* shift, const float* mean, const float* rstd, const float* drop,
               int relu, float* sums /* [2C]: dbeta, dgamma */, void* workspace, size_t workspace_bytes, void* stream);
int rbu_ag_bwd(const void* da, int64_t da_ld, const void* skip, int64_t s_ld, void* dskip, int64_t ds_ld,
               const void* yg, int64_t yg_ld, const void* yx, int64_t yx_ld, void* dyg, int64_t dyg_ld, void* dyx,
               int64_t dyx_ld, int N, int HW, int C, int F, const float* psi, const float* q0, const float* stats,
               const float* Ag, const float* Bg, const float* Ax, const float* Bx, const float* mg, const float* rg,
               const float* mx, const float* rx, const float* wpsi, float* dq, float* sums_psi, float* sums_f,
               void* workspace, size_t workspace_bytes, void* stream);
int rbu_maxpool2x2_bwd(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, void* dx, int64_t dx_ld, int N,
                       int Ho, int Wo, int C, int accumulate, void* stream);
int rbu_chan_sum(const void* x, int64_t ld, int64_t P, int C, float* out, void* workspace, size_t workspace_bytes,
                 void* stream);

/* ------------------------------------------------------------------ plain 2-class U-Net path (SURVEY.md §8f row 2)
 * `final` 1x1 convolution to two logits (train_water_segmentation.py:246,288): logits fp32 NCHW [B,2,H,W]; its
 * backward (dx bf16 view, dw [2][C], db [2]); nn.CrossEntropyLoss() on those logits (train_water_segmentation.py:304)
 * fused with the argmax confusion counts behind accuracy / IoU (:384-388, class 1 = water, ties -> class 0). */
int rbu_head2_forward(const void* x, int64_t ld, int64_t P, int HW, int C, const float* w, const float* b, float* logits,
                      void* stream);
size_t rbu_head2_backward_workspace_bytes(int64_t P, int C);
int rbu_head2_backward(const float* dlogits, const void* x, int64_t x_ld, void* dx, int64_t dx_ld, int64_t P, int HW, int C,
                       const float* w, float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream);
size_t rbu_ce2_workspace_bytes(int B, int64_t HW);
int rbu_ce2_forward(const float* logits, const int64_t* target, int B, int64_t HW, void* workspace, size_t workspace_bytes,
                    float* loss_out, int64_t* counts, void* stream);
int rbu_ce2_backward(const float* logits, const int64_t* target, int B, int64_t HW, const float* grad_out, float* dlogits,
                     void* stream);

/* ------------------------------------------------------------------ K-class heads (1 <= K <= 32)
 * RobustUNet's outc = Conv2d(b, n_classes, 1) + Sigmoid (Main_Final.py:274-277) and UNet's final = Conv2d(64, n_classes, 1)
 * trained with nn.CrossEntropyLoss (train_water_segmentation.py:246,288,304) for any class count.  RobustUNet with K = 1
 * keeps rbu_head_*, UNet with K = 2 keeps rbu_head2_* / rbu_ce2_*.  C is a power of two in [16, 256]; P % HW == 0.
 *
 * K-output 1x1 head: out[n][k][hw] = w[k].x[p] + b[k], fp32 NCHW [N][K][HW]; sigmoid != 0 applies the same
 * sigmoidf_acc as rbu_head_forward (RobustUNet outc); logits (optional) receives the pre-sigmoid values. */
int rbu_headk_forward(const void* x, int64_t ld, int64_t P, int HW, int C, int K, const float* w, const float* b,
                      int sigmoid, float* out, float* logits, void* stream);
size_t rbu_headk_backward_workspace_bytes(int64_t P, int C, int K);
/* dz = sigmoid ? dout*p*(1-p) (as rbu_head_backward) : dout;  dx = sum_k dz_k w_k (bf16 view);
 * dw[K][C] = sum_p dz x;  db[K] = sum_p dz  -- two-stage, fixed order, no float atomics */
int rbu_headk_backward(const float* dout, const float* probs, const void* x, int64_t x_ld, void* dx, int64_t dx_ld,
                       int64_t P, int HW, int C, int K, int sigmoid, const float* w, float* dw, float* db,
                       void* workspace, size_t workspace_bytes, void* stream);
/* nn.CrossEntropyLoss() over K classes + per-class argmax confusion counts [B][K][4] (TP, FP, FN, TN; ties -> lowest
 * class index, as torch.argmax); targets outside [0, K) add no loss and no counts, and are counted in *invalid.  The
 * loss is divided by B*HW.  B <= 65535. */
size_t rbu_cek_workspace_bytes(int B, int64_t HW, int K);
int rbu_cek_forward(const float* logits, const int64_t* target, int B, int64_t HW, int K, void* workspace,
                    size_t workspace_bytes, float* loss_out, int64_t* class_counts, int64_t* invalid, void* stream);
/* (softmax - onehot) * g / (B*HW); invalid pixels get 0 */
int rbu_cek_backward(const float* logits, const int64_t* target, int B, int64_t HW, int K, const float* grad_out,
                     float* dlogits, void* stream);

/* ------------------------------------------------------------------ tiled whole-scene inference
 * Sliding-window prediction at full resolution, the alternative to predict_coastline.py:386-392,583-602 (resize the
 * scene to 512², predict, scale the mask back up).  The tile grid is ny x nx tiles of th x tw; tile t = iy*nx + ix has
 * its origin at (oy[iy], ox[ix]) (DEVICE int tables).  Tile rows / columns beyond the scene are reflected with
 * F.pad(mode="reflect") semantics, so th <= 2H - 1 and tw <= 2W - 1.
 *
 * rbu_tile_gather: x fp32 NCHW [nc,H,W] -> out fp32 [Tb][nc][th][tw], tiles t0 .. t0+Tb-1. */
int rbu_tile_gather(const float* x, int nc, int H, int W, const int* oy, const int* ox, int ny, int nx, int th, int tw,
                    int t0, int Tb, float* out, void* stream);
/* rbu_tile_blend: tiles fp32 [ny*nx][K][th][tw] (1 <= K <= 32) -> labels uint8 [H,W] and, when out != NULL, the blended
 * fp32 [K][H][W].  Output row y is covered by tiles iy in [row_first[y], row_first[y] + row_count[y]), column x by
 * ix in [col_first[x], col_first[x] + col_count[x]) (DEVICE int tables); wy [th] / wx [tw] are the 1-D window weights.
 * Per pixel, over iy ascending (outer) and ix ascending (inner), each a separately rounded fp32 operation:
 *   w = wy[y - oy[iy]] * wx[x - ox[ix]];  num_k += w * v_k;  den += w;   out_k = num_k / den.
 * labels = out_0 > threshold (strict) at K = 1, else the arg-max over k (ties -> lowest k, as torch.argmax).  A gather
 * with no atomics: bit-deterministic. */
int rbu_tile_blend(const float* tiles, int K, int H, int W, const int* oy, const int* ox, int ny, int nx, int th, int tw,
                   const int* row_first, const int* row_count, const int* col_first, const int* col_count,
                   const float* wy, const float* wx, float threshold, float* out, uint8_t* labels, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RBUNET_H_ */
