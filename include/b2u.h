/* b2u.h — C-ABI of the B200-native U-Net hot path (libb2u.so).
 *
 * The reference (LUP-LuftbildUmweltPlanung/UNet) has no FFI of its own: its hot path is fastai/PyTorch module calls
 * issued from train.py:98-160 (unet_learner_MS -> DynamicUnet), train.py:246-250 (fit_one_cycle -> fwd/bwd/step) and
 * predict.py:191-337 (learn.predict per tile, numpy merge).  Each entry point below replaces the third-party ATen/cuDNN
 * call those lines reach; the exact call each one stands in for is named on the declaration.
 *
 * Conventions
 *   - plain pointers and sizes only; every buffer is owned by the caller (the Python host allocates through torch);
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns without host sync;
 *   - return 0 on success, a negative b2u_status otherwise; b2u_last_error() returns a thread-local message;
 *   - activations are NHWC bf16 with a channel pitch that is a multiple of 8 ("Cp"), weights are bf16
 *     [Cout][taps][CinP]; master parameters / gradients are fp32 in the torch layout [Cout][Cin][kh][kw].
 */
#ifndef B2U_H_
#define B2U_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum b2u_status {
  B2U_OK = 0,
  B2U_ERR_ARG = -1,      /* bad descriptor / unsupported shape */
  B2U_ERR_CUDA = -2,     /* a CUDA runtime/driver call failed  */
  B2U_ERR_NO_DEVICE = -3 /* no sm_100 device                    */
} b2u_status;

const char* b2u_last_error(void);
int b2u_version(void);
/* 0 when the current device is sm_100 and the driver entry points resolve. */
int b2u_device_check(void);

/* A strided NHWC window onto a bf16 tensor: element (n,y,x,c) lives at ptr[n*sN + y*sH + x*sW + c].
 * Plain tensors, channel slices of a concat buffer and stride-2 parity planes are all expressed this way.
 * Padding rule: the lanes from C up to round_up(C,16) (or round_up(C,8) when sW is smaller) of every pixel belong to
 * the view; kernels read them as data (so they must hold zeros in GEMM operands) and write them as zeros.  This keeps
 * every TMA row a whole number of 32-byte sectors — a row ending inside a sector halves TMA throughput. */
typedef struct b2u_view {
  void* ptr;
  int32_t C, W, H, N;
  int64_t sW, sH, sN; /* in elements; each must be a multiple of 8 (16-byte TMA stride rule) */
} b2u_view;

#define B2U_MAX_TAPS 16
#define B2U_MAX_VIEWS 4

enum {
  B2U_EPI_RELU = 1,    /* max(v, 0) */
  B2U_EPI_STATS = 2,   /* emit per-channel sum / sum-of-squares partials of the stored values */
  B2U_EPI_OUT_F32 = 4, /* store fp32 to out_f32 (dense NHWC with pitch out_f32_ld) instead of bf16 through `out` */
  /* fused 1x1 head (layers.12 of the DynamicUnet, ConvLayer(ni, n_out, ks=1, act_cls=None)): on top of the normal bf16
   * output the epilogue writes out_f32[pixel][k] = head_b[k] + sum_c head_w[k][c] * bf16(out[pixel][c]) for k < head_n
   * (<= 8), head_w being the head's staged bf16 weights [head_n][head_ld].  One pass instead of re-reading the largest
   * activation of the network.  Needs Cout <= 256 (one N tile). */
  B2U_EPI_HEAD = 8,
  B2U_EPI_HEAD_ONLY = 16 /* with B2U_EPI_HEAD: skip the bf16 output altogether (inference: nothing else reads it) */
};

/* Optional fused BatchNorm finalize of a B2U_EPI_STATS convolution (training-mode nn.BatchNorm2d statistics, what
 * b2u_bn_finalize computes in a launch of its own): the LAST CTA of the launch to retire sums the per-CTA partial rows
 * in a fixed order (double accumulation) and writes mean / invstd / scale = gamma*invstd / shift = beta - mean*scale and
 * the running statistics.  Enabled when `counter` is non-NULL: a zero-initialised uint32 owned by the caller (one per
 * plan), which the kernel leaves at zero again.  Only honoured when the partials are accumulated on chip
 * (info.fused_finalize == 1: Cout <= 512 and stats_ld <= 512); otherwise the caller runs b2u_bn_finalize. */
typedef struct b2u_bn_fin {
  uint32_t* counter;
  double count;       /* elements per channel = N*H*W of the output */
  const float* gamma; /* nullable (1) */
  const float* beta;  /* nullable (0) */
  float eps, momentum;
  float* running_mean; /* nullable */
  float* running_var;
  float* mean;
  float* invstd;
  float* scale;
  float* shift;
} b2u_bn_fin;

/* Implicit-GEMM convolution:  out[n,y,x,co] = epi( sum_t sum_ci a[tap_a[t]][n, y+tap_dy[t], x+tap_dx[t], ci] * w[co][tap_w[t]][ci] ).
 * Out-of-range reads are zero (the conv padding).  The same descriptor expresses
 *   - fprop 3x3/1x1 stride 1          (F.conv2d reached from fastai ConvLayer, train.py:141 DynamicUnet),
 *   - fprop stride 2 (taps address the four stride-2 parity planes of the input),
 *   - AvgPool2d(2)+1x1 idpath conv     (four taps, one per parity plane, weights pre-scaled by 1/4),
 *   - dgrad (conv of dY with the flipped/transposed filter; stride 2 = four launches writing parity planes of dX),
 * i.e. cudnnConvolutionForward / cudnnConvolutionBackwardData in the reference stack (SURVEY 2.1).
 * epilogue: v = acc*scale[co] + shift[co]; v += res (times (res_mask>0) if given); ReLU; v = (zmask>0) ? v : 0. */
typedef struct b2u_conv_desc {
  b2u_view a[B2U_MAX_VIEWS];
  int32_t num_a;
  b2u_view out;      /* geometry (N,H,W) defines the GEMM M space; C = Cout */
  const void* w;     /* bf16 [w_rows][w_taps][w_cinp] */
  int32_t w_rows, w_taps, w_cin, w_cinp;
  int32_t num_taps;
  int8_t tap_a[B2U_MAX_TAPS], tap_dy[B2U_MAX_TAPS], tap_dx[B2U_MAX_TAPS], tap_w[B2U_MAX_TAPS];
  const float* scale; /* nullable, per output channel; must be readable up to round_up(Cout,32) floats, 16B aligned */
  const float* shift; /* nullable (bias, or folded BN shift); same padding rule */
  b2u_view res;       /* ptr NULL = none */
  b2u_view res_mask;  /* ptr NULL = none */
  b2u_view zmask;     /* ptr NULL = none */
  uint32_t flags;
  float* stats;       /* B2U_EPI_STATS: [info.stats_rows][2][stats_ld] fp32 partials (zero-initialised by the caller) */
  int32_t stats_ld;
  float* out_f32;     /* B2U_EPI_OUT_F32 */
  int32_t out_f32_ld;
  b2u_bn_fin fin;     /* counter NULL = no fused finalize */
  /* num_out > 1: the output channels are split into num_out equal N tiles (Cout / num_out, a multiple of 16) and N
   * tile i is stored to out_nt[i] (channels 0..) instead of `out` - e.g. the four (i,j) phases of a PixelShuffle land
   * directly in the four stride-2 parity planes of the upsampled tensor (fastai PixelShuffle_ICNR without blur).
   * `out` still gives the GEMM geometry (N,H,W) and the total channel count. */
  int32_t num_out;
  b2u_view out_nt[4];
  /* w_batch_rows > 0: BATCHED weights - image n of the GEMM space multiplies rows [n * w_batch_rows, n * w_batch_rows +
   * w_rows) of `w` (which then holds out.N * w_batch_rows rows): out[n,p,r] = sum_c a[n,p,c] * w[n * w_batch_rows + r][c].
   * This is torch.bmm(A, B^T) on the implicit-GEMM kernel - the batched products of fastai's SelfAttention
   * (`bmm(f^T, g)`, `bmm(h, beta)` and their backward; reference train.py:142, params_and_main.py:83).  Pixel tiles never
   * cross an image and CTA pairs are off in this mode.  Needs a 1x1 tap table. */
  int32_t w_batch_rows;
  /* B2U_EPI_HEAD */
  const void* head_w;   /* bf16 [head_n][head_ld], channel order of this convolution's output */
  const float* head_b;  /* fp32 [head_n], nullable */
  int32_t head_n, head_ld;
} b2u_conv_desc;

typedef struct b2u_conv_info {
  int32_t m_tiles, n_tiles, block_n, tile_w, tile_h, tile_n, stages, k_chunks, grid;
  int32_t stats_rows; /* rows of the stats partial buffer: 1 per CTA (on-chip accumulation) or 4 per M tile */
  int32_t fused_finalize; /* 1: this plan runs the BatchNorm finalize itself (desc.fin honoured) */
} b2u_conv_info;

typedef struct b2u_conv_plan b2u_conv_plan;
int b2u_conv_query(const b2u_conv_desc* d, b2u_conv_info* info);
int b2u_conv_plan_create(const b2u_conv_desc* d, b2u_conv_plan** plan);
int b2u_conv_plan_info(const b2u_conv_plan* plan, b2u_conv_info* info);
int b2u_conv_run(const b2u_conv_plan* plan, void* stream);
void b2u_conv_plan_destroy(b2u_conv_plan* plan);

/* Weight gradient: dw[co][t][ci] = sum_{n,y,x} dy[n,y,x,co] * a[tap_a[t]][n, y+tap_dy[t], x+tap_dx[t], ci]
 * (cudnnConvolutionBackwardFilter in the reference stack), optionally with db[co] = sum dy[n,y,x,co].
 * Partials over `splits` pixel ranges land in `partial` (fp32 [splits][taps][co_pad][ci_pad]); b2u_wgrad_reduce sums
 * them in a fixed order (deterministic) into the torch-layout fp32 gradient. */
typedef struct b2u_wgrad_desc {
  b2u_view dy;
  b2u_view a[B2U_MAX_VIEWS];
  int32_t num_a;
  int32_t num_taps;
  int8_t tap_a[B2U_MAX_TAPS], tap_dy[B2U_MAX_TAPS], tap_dx[B2U_MAX_TAPS];
  int32_t Cout, Cin;
  int32_t want_bias;
  float* partial;        /* workspace, size from b2u_wgrad_query */
  size_t partial_bytes;
} b2u_wgrad_desc;

typedef struct b2u_wgrad_info {
  int32_t splits, co_pad, ci_pad, taps_per_unit, units, grid, k_steps, block_n, stages;
  size_t partial_bytes;
} b2u_wgrad_info;

typedef struct b2u_wgrad_plan b2u_wgrad_plan;
int b2u_wgrad_query(const b2u_wgrad_desc* d, b2u_wgrad_info* info);
int b2u_wgrad_plan_create(const b2u_wgrad_desc* d, b2u_wgrad_plan** plan);
int b2u_wgrad_run(const b2u_wgrad_plan* plan, void* stream);
void b2u_wgrad_plan_destroy(b2u_wgrad_plan* plan);

/* Sum split partials into torch-layout gradients.  dw[co_map(co)][ci][tap_kidx[t]] (+)= alpha * sum_s partial[s][t][co][ci];
 * several taps may map to the same kernel index (the fused AvgPool idpath: 4 taps -> 1 kernel element).
 * row_perm (nullable, int32[Cout]) maps GEMM row -> torch output channel (PixelShuffle-friendly row order).
 * db (nullable) receives the bias gradient. */
int b2u_wgrad_reduce(const float* partial, int32_t splits, int32_t taps, int32_t co_pad, int32_t ci_pad, int32_t Cout,
                     int32_t Cin, int32_t ksize /* kh*kw of the torch weight */, const int32_t* tap_kidx,
                     const int32_t* row_perm, float alpha, float* dw, float* db, int32_t has_bias_cols, void* stream);

/* ---- weight staging: fp32 master [Cout][Cin][kh*kw] -> bf16 GEMM layouts, all layers in ONE launch ------------- */
/* fprop layout  wf[row(co)][t][ci]        = scale * w[co][ci][t]
 * dgrad layout  wd[ci][kk-1-t][row(co)]   = scale * w[co][ci][t]   (flipped taps, transposed channels; if wd != NULL)
 * bias_rows[row(co)] = bias[co]; row(co) = row_of_co[co] if given (PixelShuffle-friendly row order), else co.
 * `items_dev` is a device array; block_start is the exclusive prefix sum of ceil(Cout/32)*ceil(Cin/32) over the items
 * (one 256-thread block per 32x32 channel tile, all taps; kk <= 9). */
typedef struct b2u_wstage_item {
  const float* w;
  const float* bias;
  const int32_t* row_of_co;
  void* wf;
  void* wd;
  float* bias_rows;
  int32_t Cout, Cin, kk, wf_cinp, wd_coutp;
  float scale;
  int32_t block_start;
  const float* dscale;   /* nullable: device scalar multiplied on top of `scale` (1/sigma of a spectral-normed weight) */
} b2u_wstage_item;
int b2u_stage_weights(const b2u_wstage_item* items_dev, int32_t n_items, int32_t total_blocks, void* stream);

/* ---- BatchNorm (training): statistics finalize / apply / backward ------------------------------------------------
 * nn.BatchNorm2d reached from fastai ConvLayer / BatchNorm (train.py:128 create_body, :141 DynamicUnet).
 * Every tensor carries its own channel pitch so that channel slices of a concat buffer can be used in place. */
/* per-channel sum / sum-of-squares partial rows [rows][2][part_ld] of a bf16 NHWC tensor (one row per block) */
int b2u_bn_stats(const void* x, int32_t ldx, int64_t pixels, int32_t C, float* partial, int32_t rows, int32_t part_ld,
                 void* stream);
/* partial rows -> mean/invstd, scale = g*invstd, shift = b - mean*scale; running stats updated with `momentum`
 * (unbiased variance) as torch does. count = elements per channel. scratch: >= ceil(rows/128)*2*ld floats (+ one more
 * level when rows > 16384); unused when rows <= 128. */
int b2u_bn_finalize(const float* partial, int32_t rows, int32_t ld, int32_t C, double count, const float* gamma,
                    const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                    float* mean, float* invstd, float* scale, float* shift, float* scratch, size_t scratch_floats,
                    void* stream);
/* eval-mode affine from running statistics */
int b2u_bn_eval_affine(int32_t C, const float* gamma, const float* beta, const float* running_mean,
                       const float* running_var, float eps, float* scale, float* shift, void* stream);
/* y = act( x*scale+shift  [+ r*rscale+rshift | + r] ) */
int b2u_bn_apply(const void* x, int32_t ldx, const float* scale, const float* shift, const void* r, int32_t ldr,
                 const float* rscale, const float* rshift, int32_t relu, void* y, int32_t ldy, int64_t pixels,
                 int32_t C, void* stream);
/* backward reductions: g = dz * mask, mask = (y>0) if y given, else (x*scale+shift>0) if relu, else 1
 * partial[row][0][c] = sum g, partial[row][1][c] = sum g*xhat  (xhat = (x-mean)*invstd) */
int b2u_bn_bwd_reduce(const void* dz, int32_t lddz, const void* x, int32_t ldx, const void* y, int32_t ldy,
                      const float* scale, const float* shift, const float* mean, const float* invstd, int32_t relu,
                      int64_t pixels, int32_t C, float* partial, int32_t rows, int32_t part_ld, void* stream);
/* dgamma = sum g*xhat, dbeta = sum g; mean_g / mean_gx feed the apply pass */
int b2u_bn_bwd_finalize(const float* partial, int32_t rows, int32_t part_ld, int32_t C, double count, float* dgamma,
                        float* dbeta, float* mean_g, float* mean_gx, float* scratch, size_t scratch_floats,
                        void* stream);
/* dx (+)= gamma*invstd*(g - mean_g - xhat*mean_gx) */
int b2u_bn_bwd_apply(const void* dz, int32_t lddz, const void* x, int32_t ldx, const void* y, int32_t ldy,
                     const float* scale, const float* shift, const float* mean, const float* invstd,
                     const float* gamma, const float* mean_g, const float* mean_gx, int32_t relu, int32_t accumulate,
                     void* dx, int32_t lddx, int64_t pixels, int32_t C, void* stream);

/* b2u_bn_bwd_reduce + b2u_bn_bwd_finalize + b2u_bn_bwd_apply in ONE launch (an in-kernel grid barrier separates the two
 * passes; the second pass re-reads dz/x from L2 when they fit).  partial: [rows][2][part_ld] scratch; sync: two
 * zero-initialised uint32 owned by the caller (arrive counter, generation), reusable across launches on one stream. */
int b2u_bn_bwd_fused(const void* dz, int32_t lddz, const void* x, int32_t ldx, const void* y, int32_t ldy,
                     const float* scale, const float* shift, const float* mean, const float* invstd,
                     const float* gamma, int32_t relu, int32_t accumulate, void* dx, int32_t lddx, int64_t pixels,
                     int32_t C, float* partial, int32_t rows, int32_t part_ld, double count, float* dgamma,
                     float* dbeta, float* mean_g, float* mean_gx, uint32_t* sync, void* stream);

/* ---- pooling ------------------------------------------------------------------------------------------------ */
/* nn.MaxPool2d(3, stride 2, padding 1) (xresnet stem, body child 3); idx = argmax position 0..8 (uint8, pitch ld),
 * first maximum wins as in ATen */
int b2u_maxpool_fwd(const void* x, void* y, uint8_t* idx, int32_t N, int32_t H, int32_t W, int32_t C, int32_t ld,
                    void* stream);
int b2u_maxpool_bwd(const void* dy, const uint8_t* idx, void* dx, int32_t accumulate, int32_t N, int32_t H, int32_t W,
                    int32_t C, int32_t ld, void* stream);

/* ---- decoder glue: PixelShuffle_ICNR (+blur) + skip BN + concat + ReLU (fastai UnetBlock.forward) ---------------
 * u: conv1x1 output, bf16 [N,h,w,ldu>=4*cu] with channel order (i,j,c) (rows permuted at weight staging);
 * skip: bf16 [N,2h,2w,lds]; cat: bf16 [N,2h,2w,ldc]: channels [0,cu) = blur(shuffle(u)) (blur=0: plain shuffle),
 * [cu,cu+cs) = act(skip*sscale+sshift) (sscale NULL: copy, e.g. the network input of MergeLayer(dense=True)),
 * remaining lanes zero.  cu must be a multiple of 8. */
int b2u_shuffle_cat_fwd(const void* u, int32_t ldu, int32_t cu, int32_t blur, const void* skip, int32_t lds,
                        int32_t cs, const float* sscale, const float* sshift, int32_t skip_relu, void* cat,
                        int32_t ldc, int32_t N, int32_t h, int32_t w, void* stream);
/* backward of the shuffle(+blur) part: du[n,h,w,(i,j,c)] = (u>0) * blur^T(dcat[..., 0:cu]) */
int b2u_shuffle_bwd(const void* dcat, int32_t ldc, const void* u, void* du, int32_t ldu, int32_t cu, int32_t blur,
                    int32_t N, int32_t h, int32_t w, void* stream);
/* the same without blur, with the ReLU mask taken from the upsampled tensor itself (cat[n,2y+i,2x+j,c] = relu(u[...])),
 * so that the pre-shuffle activation need not exist (the conv stores its phases straight into the parity planes) */
int b2u_shuffle_bwd_from_cat(const void* dcat, const void* cat, int32_t ldc, void* du, int32_t ldu, int32_t cu,
                             int32_t N, int32_t h, int32_t w, void* stream);
/* odd skip sizes (e.g. the reference's default 400-px tiles: 25 -> 13 -> 26 vs 25): the concat / its gradient is
 * [N,Ho,Wo,ldc] with Ho in {2h, 2h-1}, Wo in {2w, 2w-1} - the last row / column of the upsampled tensor is cropped,
 * which is what fastai's F.interpolate(up_out, skip.shape[-2:], mode='nearest') computes for 2h -> 2h-1 */
int b2u_shuffle_cat_fwd_crop(const void* u, int32_t ldu, int32_t cu, int32_t blur, const void* skip, int32_t lds,
                             int32_t cs, const float* sscale, const float* sshift, int32_t skip_relu, void* cat,
                             int32_t ldc, int32_t N, int32_t h, int32_t w, int32_t Ho, int32_t Wo, void* stream);
int b2u_shuffle_bwd_crop(const void* dcat, int32_t ldc, const void* u, void* du, int32_t ldu, int32_t cu, int32_t blur,
                         int32_t N, int32_t h, int32_t w, int32_t Ho, int32_t Wo, void* stream);
/* replicate the last row / column of an NHWC bf16 tensor (pitch ld) to even extents, and the adjoint: with it the
 * 2x2 mean folded into the idpath 1x1 convolution equals nn.AvgPool2d(2, ceil_mode=True) on odd sizes (fastai ResBlock) */
int b2u_pad_even_fwd(const void* x, void* xp, int32_t ld, int32_t N, int32_t H, int32_t W, void* stream);
int b2u_pad_even_bwd(const void* dxp, void* dx, int32_t accumulate, int32_t ld, int32_t N, int32_t H, int32_t W,
                     void* stream);
/* dst[p][dst_off .. dst_off+lanes) = src[p][src_off .. src_off+lanes) for `pixels` pixels (lanes, offsets and pitches
 * multiples of 8): fastai MergeLayer(dense=True) `torch.cat([x, input], dim=1)` of the final stage (unet.py layers.10) */
int b2u_copy_lanes(const void* src, int32_t lds, int32_t src_off, void* dst, int32_t ldd, int32_t dst_off,
                   int32_t lanes, int64_t pixels, void* stream);

/* out[p,c] = (z[p,c] > 0 ? 1 : 0) * sum_{k<K} a[p,k] * w[c][k], K <= 8, all bf16 (z nullable): the input gradient of the 1x1
 * head conv (GEMM K = number of classes), i.e. cudnnConvolutionBackwardData for layers.12 of the DynamicUnet.  w is the
 * dgrad weight layout [C][ldw] produced by b2u_stage_weights. */
int b2u_pointwise_smallk(const void* a, int32_t lda, int32_t K, const void* w, int32_t ldw, const void* z, int32_t ldz,
                         void* out, int32_t ldo, int64_t pixels, int32_t C, void* stream);

/* ---- layout casts at the API edge --------------------------------------------------------------------------- */
/* Input contract (A0): the reference reads every GeoTIFF dtype as int32 -> float32 (data.py:18-28), 16-bit datasets
 * (utils.py:72-89 get_datatype 'int16') are divided by 255 inside its batch transform (utils.py:248-249, 288-289) and
 * everything is divided by 255 by fastai's IntToFloatTensor (MaskBlock, data.py:100); the regression variant
 * (RegressionBlock, data.py:98) skips IntToFloatTensor.  x_dtype: element type of the source; value = (raw / div) / div2
 * in fp32 (uint8 tiles: div 255, div2 1; 16-bit datasets: 255, 255; fp32 already scaled: 1, 1). */
#define B2U_DT_F32 0
#define B2U_DT_U8 1
#define B2U_DT_U16 2
#define B2U_DT_I16 3
/* x NCHW of x_dtype -> bf16 NHWC pitch ld, channels [ch_off, ch_off+write_c) written (lanes >= C zeroed) */
int b2u_nchw_to_nhwc(const void* x, int32_t x_dtype, float div, float div2, void* y, int32_t N, int32_t C, int32_t H,
                     int32_t W, int32_t ld, int32_t ch_off, int32_t write_c, void* stream);
/* im2col of an NHWC bf16 tensor with few channels: y[n,oy,ox, c*ks*ks + ky*ks + kx] = x[n, oy*stride+ky-pad, ox*stride+kx-pad, c]
 * (zeros outside the image and in lanes C*ks*ks .. ldy; the channel order of torch.nn.functional.unfold and of a conv
 * weight [Cout][Cin][kh][kw] read as rows of Cin*kh*kw).  Used for the first stem convolution (xresnet.py stem: 3x3
 * stride 2 over the n_in image bands, reached from train.py:98-160 `unet_learner_MS`): over the 36 im2col lanes it is a
 * 1x1 convolution with whole-sector rows, and so is its weight gradient. */
int b2u_im2col(const void* x, int32_t ldx, int32_t C, int32_t N, int32_t H, int32_t W, int32_t ks, int32_t stride,
               int32_t pad, void* y, int32_t ldy, void* stream);
/* tile t = raster[:, y0[t]:y0[t]+P, x0[t]:x0[t]+P] / div / div2 -> bf16 NHWC [T,P,P,ld]: the crop of
 * create_tiles_unet.py:410 fused with the input contract above and the layout cast; raster is [C][Y][X] of r_dtype on
 * the device */
int b2u_crop_tiles(const void* raster, int32_t r_dtype, float div, float div2, int32_t C, int64_t Y, int64_t X,
                   const int32_t* y0, const int32_t* x0, int32_t T, int32_t P, void* out, int32_t ld, void* stream);
/* Training batch cut out of a device-resident raster and its label raster, with the dihedral augmentation in the same
 * pass: the crop of create_tiles_unet.py:410 (the image and mask tiles split_raster writes) and the flips / 90-degree
 * rotations of utils.py:196-295 (SegmentationAlbumentationsTransform on image and mask together).
 *   x[t][c] = D_op[t](raster[c, y0[t]:y0[t]+P, x0[t]:x0[t]+P])      raw band values of r_dtype (B2U_DT_U8/U16/I16)
 *   y[t]    = D_op[t](labels[y0[t]:y0[t]+P, x0[t]:x0[t]+P])          l_dtype B2U_DT_U8 (class ids) or B2U_DT_F32
 * raster [C][Y][X], labels [Y][X]; y0 / x0 / op are device int32 [T].  D_op flips the last axis when op & 4, then turns
 * op & 3 quarter turns as torch.rot90(., k, (-2, -1)); op 0 is the identity.  Pixels outside the raster are zero. */
int b2u_crop_train_batch(const void* raster, int32_t r_dtype, int32_t C, int64_t Y, int64_t X, const void* labels,
                         int32_t l_dtype, const int32_t* y0, const int32_t* x0, const int32_t* op, int32_t T, int32_t P,
                         void* x, void* y, void* stream);
/* bf16/f32 NHWC -> fp32 NCHW */
int b2u_nhwc_to_nchw_f32(const void* x, int32_t x_is_f32, int32_t ld, float* y, int32_t N, int32_t C, int32_t H,
                         int32_t W, void* stream);

/* ---- loss: CrossEntropyLossFlat(axis=1) with class weights, mean reduction (train.py:195,211) ----------------- */
/* logits fp32 [P][ld]; labels uint8 [P]; wsum = sum_p weight[label_p] (b2u_ce_weight_sum first, `rows` block partials).
 * b2u_ce_fwd_bwd writes dlogits bf16 [P][ldg] = grad_scale*w[y]*(softmax - onehot)/wsum (NULL: loss only) and block
 * partials of sum w[y]*nll; b2u_ce_finalize: loss = sum(loss_partial)/sum(wsum_partial). */
int b2u_ce_weight_sum(const uint8_t* labels, int64_t P, const float* weight, int32_t C, float* wsum_partial,
                      int32_t rows, void* stream);
int b2u_ce_fwd_bwd(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C, const float* weight,
                   const float* wsum_partial, int32_t wsum_rows, void* dlogits, int32_t ldg, float* loss_partial,
                   int32_t rows, float grad_scale, void* stream);
int b2u_ce_finalize(const float* loss_partial, int32_t rows, const float* wsum_partial, int32_t wsum_rows, float* loss,
                    void* stream);

/* ---- loss: fastai FocalLossFlat(axis=1, gamma, weight) -------------------------------------------------------- */
/* logits / labels / dlogits as for CE.  Per pixel l = w[y]*nll, f = (1-exp(-l))^gamma * l; `rows` block partials of
 * sum f, reduced by b2u_mse_finalize(P) for mean (mean != 0) or b2u_mse_finalize(1) for sum.  dlogits (NULL: loss only)
 * = df/dlogits * grad_scale (/ P for mean).  gamma >= 0. */
int b2u_focal_fwd_bwd(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C, const float* weight,
                      float gamma, int32_t mean, void* dlogits, int32_t ldg, float* loss_partial, int32_t rows,
                      float grad_scale, void* stream);
/* ---- loss: fastai DiceLoss(axis=1, smooth, reduction, square_in_union), two phases ---------------------------- */
/* Samples are N runs of HW pixels.  b2u_dice_stats writes fp32 partial[N][blocks_per_sample][3][C] = per block
 * {sum p*t, sum p (sum p^2 with square_in_union), sum t}.  b2u_dice_bwd folds them per (n, c) in block order,
 * writes loss_partial[n] = sum_c (1 - (2I+s)/(U+s)) and dlogits (NULL: loss only) = d(loss)/d(logits) * grad_scale
 * (/ (N*C) for mean); the loss is b2u_mse_finalize(loss_partial, N, mean ? N*C : 1).  Deterministic, no atomics. */
int b2u_dice_stats(const float* logits, int32_t ld, const uint8_t* labels, int32_t N, int64_t HW, int32_t C,
                   int32_t square_in_union, float* partial, int32_t blocks_per_sample, void* stream);
int b2u_dice_bwd(const float* logits, int32_t ld, const uint8_t* labels, int32_t N, int64_t HW, int32_t C,
                 int32_t square_in_union, const float* partial, int32_t blocks_per_sample, float smooth, int32_t mean,
                 void* dlogits, int32_t ldg, float* loss_partial, float grad_scale, void* stream);

/* ---- regression variant: MSELossFlat(axis=1) (train.py:189-192) + the sums behind fastai's rmse / R2Score metrics -- */
/* pred = lane 0 of the fp32 head output [P][ld]; target fp32 [P]; loss = mean (pred - target)^2; dpred bf16 [P][ldg]
 * (NULL: loss only) lane 0 = grad_scale * 2 (pred - target) / P, other lanes 0.  `rows` block partials, then finalize. */
int b2u_mse_fwd_bwd(const float* pred, int32_t ld, const float* target, int64_t P, void* dpred, int32_t ldg,
                    float* loss_partial, int32_t rows, float grad_scale, void* stream);
int b2u_mse_finalize(const float* loss_partial, int32_t rows, int64_t P, float* loss, void* stream);
/* sums[0..3] (device, double) += {sum (pred-target)^2, sum target, sum target^2, P}; partial: rows*3 doubles of scratch;
 * ticket: one zero-initialised uint32.  Fixed-order combination (deterministic). */
int b2u_regression_sums(const float* pred, int32_t ld, const float* target, int64_t P, double* partial, int32_t rows,
                        double* sums, uint32_t* ticket, void* stream);
/* ---- validation metric DiceMulti (train.py:196): counts (device, uint64 [3*C]) += per class {#(pred==c & y==c),
 * #(pred==c), #(y==c)} with pred = argmax_c logits (first maximum wins); Dice_c = 2 I_c / (P_c + T_c). */
int b2u_dice_counts(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C, uint64_t* counts,
                    void* stream);

/* ---- optimizer ------------------------------------------------------------------------------------------------ */
/* ---- data-parallel gradient exchange: the fp32 gradient range is cast to bf16 for the NCCL all-reduce (half the bytes
 * over NVLink) and back before the optimizer.  x / y: fp32 ranges 16-byte aligned, bf16 ranges 8-byte aligned. */
int b2u_cast_f32_bf16(const float* x, void* y, int64_t n, void* stream);
int b2u_cast_bf16_f32(const void* x, float* y, int64_t n, void* stream);

/* p -= lr * grad_scale * g over one flat fp32 buffer (BASELINE config 1: plain SGD) */
int b2u_sgd_step(float* p, const float* g, int64_t n, float lr, float grad_scale, void* stream);
/* fastai Adam (train.py:218): decoupled wd, per-segment lr / wd via device tables (seg_end = exclusive end offsets);
 * hyper (device, 6 floats) = {mom, sqr_mom, eps, 1-mom^step, 1-sqr_mom^step, grad_scale} so that the one-cycle
 * schedule can change them between replays of a captured graph. */
int b2u_adam_step(float* p, const float* g, float* m, float* v, int64_t n, const int64_t* seg_end, const float* seg_lr,
                  const float* seg_wd, int32_t nseg, const float* hyper, void* stream);

/* ---- prediction: softmax + overlap-tile accumulate, normalise + argmax (predict.py:284-334) ------------------- */
/* logits fp32 [T][th][tw][ld]; tile t sits at (y0[t], x0[t]) of the full raster; acc fp32 [C][Y][X] and cnt uint8
 * [Y][X] cover the raster window starting at (y_off, x_off).  The launch adds the first min(*n_sel_dev, max_sel)
 * tiles listed in `sel` (0 < max_sel <= T); the count lives on the device, so the host can refill a batch's tile
 * origins and class lists with one device copy instead of waiting for them.  Tiles within one launch must not overlap
 * each other (the host colours the overlap graph), which makes the sums independent of scheduling without atomics.
 * mode 0: softmax probabilities are added.  mode 1: the `large_file` merge (predict.py:217-219): every probability is
 * quantised to np.around(p * 31) (int8 in the reference; the sums <= 4*31 are exact in the fp32 accumulator).
 * mode 2: the regression merge (predict.py:196-198, 300-302): the raw network output is added, no softmax. */
int b2u_stitch_accumulate(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                          const int32_t* y0, const int32_t* x0, const int32_t* sel, const int32_t* n_sel_dev,
                          int32_t max_sel, int32_t mode, float* acc, uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off,
                          int64_t x_off, void* stream);
/* mask[y][x] = argmax_c acc[c][y][x]/cnt (first max wins like np.argmax, unplaced pixels -> 0), uint8.  int_div != 0:
 * the quotients are floored first, as the `large_file` merge floor-divides its int8 sums (predict.py:318-323). */
int b2u_stitch_finalize(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X, int32_t int_div,
                        uint8_t* mask, void* stream);
/* out[c][y][x] = acc/cnt where tiles were placed, `nodata` elsewhere (regression: -9999, predict.py:313-316; also the
 * averaged probabilities of the `all_classes` / `specific_class` merge, predict.py:326-337, nodata 0) */
int b2u_stitch_finalize_mean(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X, float nodata,
                             float* out, void* stream);
/* The averaged class probabilities of the `all_classes` / `specific_class` merge (predict.py:226-254, 307-337) for
 * classes [c0, c0 + nc) over columns [x0, x0 + w) of acc / cnt, written pixel-interleaved - the sample order of a
 * striped GeoTIFF: out[y * pitch + (x - x0) * nc + k] for y < Y, pitch in elements (>= w * nc), 1 <= nc <= 32.
 * mode 0 (sums of accumulate mode 0): fp32 acc / cnt, the same IEEE division as b2u_stitch_finalize_mean, 0 where
 * cnt == 0.  mode 1 (sums of accumulate mode 1, `large_file`): int8, the reference's int8 arithmetic - the sum wraps
 * modulo 256 and is floor-divided (toward -inf) by the count as int8 where that is > 0; 0 where cnt == 0. */
int b2u_stitch_finalize_probs(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X, int32_t c0,
                              int32_t nc, int64_t x0, int64_t w, int32_t mode, void* out, int64_t pitch, void* stream);
/* per-tile softmax probabilities (fp32 NCHW, what learn.predict returns, predict.py:193-203) and argmax */
int b2u_softmax_nchw(const float* logits, int32_t ld, int32_t C, int64_t tiles, int32_t H, int32_t W, float* probs,
                     uint8_t* argmax, void* stream);

/* ---- assessment: confusion counts of predicted class maps against truth maps (predict.py:56-143 validation_vision,
 * sklearn.metrics.confusion_matrix / classification_report) -------------------------------------------------------
 * T images of H x W uint8 class ids; pixel (t, y, x) of a map is at base + t * stride + y * pitch + x (the stride is
 * unused when T == 1; pitch and base need no alignment, rows are read with 16-byte loads where both maps allow).
 * Accumulates (device):  joint[truth * C + pred] += 1 (uint64 [C][C]) for pixels with both values < C, skipped += 1
 * (uint64) for the others; tile_hist (nullable, uint32 [T][2][C]) += per image the truth histogram ([t][0]) and the
 * prediction histogram ([t][1]) of the counted pixels.  1 <= C <= 32.  Integer counts: bit-identical on every run. */
int b2u_confusion_counts(const uint8_t* pred, int64_t pred_pitch, int64_t pred_stride, const uint8_t* truth,
                         int64_t truth_pitch, int64_t truth_stride, int32_t T, int32_t H, int32_t W, int32_t C,
                         uint64_t* joint, uint32_t* tile_hist, uint64_t* skipped, void* stream);
/* ---- assessment of regression maps: error statistics of fp32 predictions against fp32 truth ------------------------
 * Same layout as b2u_confusion_counts, in floats: pixel (t, y, x) of a map is at base + t * stride + y * pitch + x
 * (4-byte aligned; rows are read with 16-byte loads where both maps allow).  A pixel is skipped (skipped += 1, uint64)
 * when either value is not finite, the prediction equals pred_nodata or the truth equals truth_nodata (NaN: no nodata
 * value).  Over the counted pixels, with e = p - t, a record of 15 doubles holds
 *   {n, mean t, mean p, M2 t, M2 p, C tp, sum |e|, sum e, sum e^2, min t, max t, min p, max p, min e, max e}
 * (M2 = sum of squared deviations from the mean, C = sum of the products of the deviations).  `totals` (double [15]) and
 * `tile_rec` (nullable, double [T][15], one record per image) are merged with the call's records by Chan et al.'s pairwise
 * update, so they accumulate over calls; a zero-filled record is empty.  scratch: `scratch_records` >= T records of 15
 * doubles (more records allow more blocks per image); ticket: one zero-initialised uint32 that the call leaves zero.
 * Every merge happens in a fixed order, without float atomics: the records are the same bits on every run. */
int b2u_regression_assess(const float* pred, int64_t pred_pitch, int64_t pred_stride, const float* truth,
                          int64_t truth_pitch, int64_t truth_stride, int32_t T, int32_t H, int32_t W, float pred_nodata,
                          float truth_nodata, double* totals, double* tile_rec, uint64_t* skipped, double* scratch,
                          int64_t scratch_records, uint32_t* ticket, void* stream);

/* ---- SelfAttention (fastai layers.SelfAttention on UnetBlock.conv2 when self_attention=True, train.py:142) --------
 * The 1x1 query / key / value convolutions run through b2u_conv_*, the two batched attention products are plain
 * library GEMMs issued by the host layer; these entry points are the rest of the block. */
/* torch.nn.utils.spectral_norm of W fp32 [Co][Ci]: training != 0 runs ONE power iteration in place
 * (v = normalize(W^T u), u = normalize(W v), eps 1e-12); sigma_out[0] = u.(W v), sigma_out[1] = 1/sigma */
int b2u_spectral_norm(const float* W, int32_t Co, int32_t Ci, float* u, float* v, int32_t training, float* sigma_out,
                      void* stream);
/* gradient through W_sn = W / sigma(W) with u, v constant: dW <- (dW - sum(dW * W_sn) u v^T) / sigma, in place */
int b2u_spectral_norm_bwd(float* dW, const float* W, int32_t Co, int32_t Ci, const float* u, const float* v,
                          const float* sigma, void* stream);
/* batched transpose of an NHWC-style bf16 tensor: y[b][c][i] = x[b][i][c] for i < n, c < C (x rows of pitch ldx, y rows of
 * pitch ldy >= n; pad lanes of y are zeroed) - puts the contraction index of a batched product innermost */
int b2u_transpose_bnc(const void* x, int32_t ldx, void* y, int32_t ldy, int32_t B, int32_t n, int32_t C, void* stream);
/* beta[b][i][j] = softmax over i of S[b][i][j] (F.softmax(..., dim=1)), bf16 [B][n] rows of pitch ld >= n; betaT
 * (nullable, same shape) also receives the transpose betaT[b][j][i] */
int b2u_softmax_dim1(const void* S, void* beta, void* betaT, int32_t B, int32_t n, int32_t ld, void* stream);
/* dS = beta * (dbeta - sum_i beta * dbeta), column-wise; dS may alias dbeta; dST (nullable) receives the transpose */
int b2u_softmax_dim1_bwd(const void* beta, const void* dbeta, void* dS, void* dST, int32_t B, int32_t n, int32_t ld,
                         void* stream);
/* out = gamma[0] * o + x over `elems` bf16 elements (multiple of 8) */
int b2u_attn_out(const void* o, const void* x, const float* gamma, void* out, int64_t elems, void* stream);
/* d_o = gamma[0] * dout (bf16) and dgamma[0] = sum(dout * o) (fp32, fixed-order two-stage reduction;
 * scratch >= 1024 floats + 1 counter word, zero-initialised once by the caller) */
int b2u_attn_out_bwd(const void* dout, const void* o, const float* gamma, void* d_o, float* dgamma, float* scratch,
                     int64_t elems, void* stream);

/* sizeof() of the ABI structs as this library was compiled, for bindings to verify their mirrors:
 * which = 0 b2u_view, 1 b2u_conv_desc, 2 b2u_conv_info, 3 b2u_wgrad_desc, 4 b2u_wgrad_info, 5 b2u_wstage_item, 6 b2u_bn_fin */
int b2u_abi_sizeof(int which);

#ifdef __cplusplus
}
#endif
#endif /* B2U_H_ */
