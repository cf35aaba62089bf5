/*
 * x3d_b200.h -- C ABI of the B200 (sm_100a) X3D forward path.
 *
 * The reference (fcogidi/X3D-tf) has no FFI of its own: its hot path is a chain of
 * tf.keras layer calls inside model.py.  Each entry point below replaces the TensorFlow op
 * (or short chain of ops) that one of those call sites lowers to; the reference call site is
 * cited on every function.  The Python classes in x3d_tf_b200/model.py (same names and
 * constructor arguments as model.py) bind these through ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - Plain C: device pointers, sizes, a cudaStream_t passed as void*.  No torch types.
 *   - Every call is asynchronous on `stream`, never synchronises, never allocates.
 *   - Return value: 0 = ok, negative = X3D_ERR_*.  x3d_last_error() gives a thread-local text.
 *   - Activations are channels-last NDHWC, row-major, `C` = STORED channel count, which must be a
 *     multiple of 8 (the host zero-pads 54->56, 108->112 ...; padded channels carry zeros and
 *     have zero weights).  The stem's 3-channel input is the only exception.
 *   - `dtype` selects the storage type of activations: X3D_F32 or X3D_BF16.  Arithmetic is
 *     fp32-accumulate in both cases.  Weights/biases passed as `const float*` are fp32 with the
 *     inference BatchNorm already folded in (scale into the kernel, shift as bias).
 *   - 64-bit element offsets are used throughout (X3D-L activations exceed 2^31 bytes).
 */
#ifndef X3D_B200_H_
#define X3D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define X3D_B200_VERSION 100

enum x3d_dtype { X3D_F32 = 0, X3D_BF16 = 1 };

enum x3d_status {
  X3D_OK = 0,
  X3D_ERR_INVALID_ARG = -1,   /* bad size / alignment / dtype / null pointer */
  X3D_ERR_UNSUPPORTED = -2,   /* shape outside what the kernel was built for */
  X3D_ERR_LAUNCH = -3,        /* CUDA reported an error at launch */
  X3D_ERR_NO_DEVICE = -4      /* no sm_100 device / driver entry point missing */
};

int x3d_version(void);
const char* x3d_last_error(void);

/* CRC-32C (Castagnoli) of a host buffer, continuing from `crc` (0 to start).  Used by the
 * TF-bundle reader that stands in for model.load_weights (train.py:137-143, eval.py:78-81). */
uint32_t x3d_crc32c(const void* data, size_t len, uint32_t crc);

/* ---- Stem: X3D_Stem.call, model.py:202-210 -------------------------------------------------
 * tf.pad(H,W by 1) -> Conv3D 1x3x3 s(1,2,2) valid -> tf.pad(T by kt/2) -> channelwise Conv3D
 * kt x1x1 -> BatchNormalization -> ReLU, as ONE kernel.
 *   in   [N,T,H,W,3]        in_dtype (X3D_F32 | X3D_BF16)
 *   ws   [3,3,3,C] fp32     conv_s kernel (dh,dw,ci,c)
 *   wt   [kt,C]   fp32      conv_t kernel with the BN scale folded in
 *   bias [C]      fp32      BN shift
 *   out  [N,T,Ho,Wo,C]      out_dtype;  Ho=(H-1)/2+1, Wo=(W-1)/2+1
 * kt must be 5 (NETWORK.C1_TEMP_FILTER of every shipped config). */
int x3d_stem_fwd(const void* in, int in_dtype, const float* ws, const float* wt,
                 const float* bias, void* out, int out_dtype,
                 int N, int T, int H, int W, int C, int kt, void* stream);

/* Same operation on the tensor cores, bf16 output (the kernel the bf16 path uses): the two convs
 * are merged into one kt x3x3 implicit GEMM (exact: nothing non-linear sits between them).
 *   wc  bf16 [kt][4][32][8]: wc[dt][k/8][c][k%8] = ws[k][c] * wt[dt][c] (BN scale folded),
 *       k = (dh*3+dw)*3+ci < 27, c < C; zero elsewhere.   C <= 32. */
int x3d_stem_tc_fwd(const void* in, int in_dtype, const void* wc, const float* bias, void* out,
                    int N, int T, int H, int W, int C, int kt, void* stream);

/* ---- Pointwise (1x1x1) convolution as a GEMM, SIMT fp32-accumulate path ---------------------
 * One entry point for Bottleneck.a+bn_a+relu (model.py:306-308), Bottleneck.c+bn_c with the
 * SE-scale/swish prologue and the residual add + ReLU of ResBlock (model.py:311-318,389-392),
 * the strided shortcut conv + bn_r (model.py:386-388), conv5 (model.py:117) and the head's
 * fc1 / fc2 (model.py:119-121).
 *   D[m, 0:Nc] = act( bias + sum_k pro(A[row(m), k]) * Wt[k, 0:Nc] (+ R[m, 0:Nc]) )
 *   A    [*, lda]   a_dtype;  row(m) = m, or for gather != 0 the input pixel
 *                   (n, t, ho*stride, wo*stride) of output pixel m = ((n*T+t)*Ho+ho)*Wo+wo
 *   Wt   [K, ldw]   fp32, BN scale folded;  bias [Nc] fp32 (may be NULL)
 *   pro(a) = a                         if se == NULL and !swish
 *          = swish(a * se[m / rows_per_clip, k])   (se NULL => factor 1; swish(x)=x*sigmoid(x))
 *   R    [M, ldr]   residual, d_dtype (may be NULL);  act = ReLU if relu else identity
 *   D    [M, ldd]   d_dtype
 * Accumulation is fp32.  fp32 in / fp32 out runs on the tensor cores with the 3xTF32 split (each
 * operand = two TF32 halves; lo.hi + hi.lo + hi.hi): fp32-level accuracy, 2e-7..4e-6 of the
 * output scale measured; bf16 activations run on CUDA cores (the tcgen05 path is x3d_pw_tc_fwd). */
typedef struct x3d_pw_args {
  const void* A; const float* Wt; const float* bias; const void* R; const float* se; void* D;
  int64_t M; int32_t K, Nc, lda, ldw, ldr, ldd;
  int64_t rows_per_clip;
  int32_t a_dtype, d_dtype, swish, relu;
  int32_t gather, T, Ho, Wo, Hi, Wi, stride;
} x3d_pw_args;
int x3d_pw_fwd(const x3d_pw_args* args, void* stream);

/* fp32 pointwise conv on the 5th-generation tensor cores (tcgen05.mma kind::tf32, TMEM accumulator,
 * TMA operands) with the 3xTF32 split -- fp32-level accuracy; the training path's GEMM (forward of
 * a / c / shortcut / conv5 / fc1 / fc2, model.py:246-253, 292-299, 360-367, 78-108, and their
 * backward-data):   D[M, Nc] = act(bias + A[M, K] . B^T)
 *   A [M, lda] fp32, K % 4 == 0;  D [M, ldd] fp32, Nc % 4 == 0;  bias [Nc] fp32 or NULL;  relu 0/1
 *   stats: NULL, or fp64 [2][Nc] (caller-zeroed) that receives += column sums and sums of squares of
 *   D -- the batch statistics of the BatchNormalization that follows the conv (model.py:254,300,89),
 *   accumulated in the epilogue instead of by a second pass over D (bias must be NULL, relu 0)
 *   Bsplit fp32 [2][Nc][K]: plane 0 = B rounded to TF32, plane 1 = B - plane 0 (B = the [Nc, K]
 *   operand with the reduction dimension contiguous), produced by
 * x3d_tf32_split(W, out, rows, cols, ld, transpose): out[.][r][c] from W[r*ld + c], or from
 *   W[c*ld + r] when transpose = 1 (forward: W is the [K, Nc] kernel, rows = Nc, cols = K, transpose;
 *   backward-data: the same kernel as stored, rows = K, cols = Nc). */
int x3d_tf32_split(const float* W, float* out, int rows, int cols, int ld, int transpose, void* stream);
int x3d_pw_tf32_fwd(const float* A, const float* Bsplit, const float* bias, float* D, int64_t M, int K,
                    int Nc, int lda, int ldd, int relu, double* stats, void* stream);
/* The same GEMM in the bf16 operand mode of the mixed-precision training step (kind::f16 MMA, fp32
 * accumulation): D = act(bias + bf16(A) . Wb^T), A rounded to bf16 (round-to-nearest-even) in shared
 * memory after the fp32 TMA load; arguments, constraints and the stats epilogue as x3d_pw_tf32_fwd.
 *   Wb bf16 [Nc][round_up(K, 8)] (padding zero), produced by
 * x3d_bf16_round(W, out, rows, cols, ld, transpose): out[r][c] = bf16_rn(W[r*ld + c]), or of
 *   W[c*ld + r] when transpose = 1, rows of pitch round_up(cols, 8) with zero padding (orientations as
 *   x3d_tf32_split). */
int x3d_bf16_round(const float* W, void* out, int rows, int cols, int ld, int transpose, void* stream);
int x3d_pw_bf16_train_fwd(const float* A, const void* Wb, const float* bias, float* D, int64_t M, int K,
                          int Nc, int lda, int ldd, int relu, double* stats, void* stream);

/* ---- Channelwise 3x3x3 convolution: Bottleneck.b + bn_b, model.py:309-310 -------------------
 * Grouped Conv3D(groups=C) stride (1,s,s), TF padding='same' (T: 1 before; H/W: pad_h/pad_w
 * before, derived on the host from TF's rule), + BN, and -- when `se_partial` != NULL -- the
 * per-clip, per-channel sums of the output that se_pool (model.py:312) needs, written as
 * fixed-order partial sums (deterministic; no atomics):
 *   in  [N,T,H,W,C]; w [27,C] fp32 (dt,dh,dw major; BN scale folded); bias [C] fp32
 *   out [N,T,Ho,Wo,C], Ho=ceil(H/s), Wo=ceil(W/s)
 *   se_partial [N, nblk, C] fp32 with nblk = x3d_dw_partial_blocks(...) (one row per spatial tile
 *   of the launch; depends on the shape and dtype only) */
int x3d_dw_partial_blocks(int T, int H, int W, int C, int stride, int dtype);
int x3d_dw3x3x3_fwd(const void* in, const float* w, const float* bias, void* out,
                    float* se_partial, int N, int T, int H, int W, int C, int stride,
                    int pad_h, int pad_w, int dtype, void* stream);
/* The same with the activation that follows bn_b fused into the epilogue: act = 1 applies swish
 * (model.py:316) to the output.  Only for blocks WITHOUT Squeeze-Excitation (se_partial must be
 * NULL): with SE the per-clip scale has to be applied before the swish, which the projection GEMM's
 * prologue does.  act = 0 is x3d_dw3x3x3_fwd. */
int x3d_dw3x3x3_act_fwd(const void* in, const float* w, const float* bias, void* out,
                        float* se_partial, int N, int T, int H, int W, int C, int stride,
                        int pad_h, int pad_w, int dtype, int act, void* stream);

/* The same layer (model.py:309-316; bf16 only) with lanes = pixels and warp = channel pair, so that the
 * 27 taps sit in uniform registers and the packed FFMA2 reads two register operands instead of three
 * (csrc/x3d_dw_planar.cu).  `taps`: device fp32 [ceil(C/2)][28][2] = per channel pair the 27 BN-folded
 * taps (dt, dh, dw major) and the BN shift, as (channel 2p, channel 2p+1); copied into the constant
 * bank, stream-ordered, by the call.  C <= 576.  se_partial [N, nblk, C], nblk =
 * x3d_dw_planar_partial_blocks(...); act as for x3d_dw3x3x3_act_fwd.  The tap table is one per device:
 * calls on ONE stream (or stream-ordered against each other) only.
 * x3d_dw_planar_lane_permille: output pixels / (pixels of the tiles that cover them) * 1000, i.e. how
 * much of the kernel's lane grid a shape uses (1000 at 64x64, 875 at 56x56); 0 = no plan. */
int x3d_dw_planar_partial_blocks(int T, int H, int W, int C, int stride);
int x3d_dw_planar_lane_permille(int T, int H, int W, int C, int stride);
int x3d_dw3x3x3_planar_fwd(const void* in, const float* taps, void* out, float* se_partial, int N, int T,
                           int H, int W, int C, int stride, int pad_h, int pad_w, int act, void* stream);

/* ---- Squeeze-Excitation MLP: se_pool/se_fc1/se_fc2, model.py:311-314 ------------------------
 *   mean[n,c] = inv_count * sum_b partial[n,b,c];  z = relu(mean.w1 + b1);  scale = sigmoid(z.w2 + b2)
 *   w1 [C,Cw], b1 [Cw], w2 [Cw,C], b2 [C] fp32;  scale [N,C] fp32.   Cw <= 64. */
int x3d_se_mlp_fwd(const float* partial, int nblk, float inv_count, const float* w1,
                   const float* b1, const float* w2, const float* b2, float* scale,
                   int N, int C, int Cw, void* stream);

/* ---- Global average pool: AdaptiveAvgPool3D.call, model.py:473-483 --------------------------
 *   in [N,P,C] dtype -> out [N,C] fp32 (mean over the P = T*H*W positions), fixed order. */
int x3d_avgpool_fwd(const void* in, float* out, int N, int64_t P, int C, int dtype, void* stream);

/* ---- Softmax (fp32) + view average: model.py:122-127 ----------------------------------------
 *   logits [N,ncls] fp32 -> probs [N/num_preds, ncls] fp32; num_preds consecutive rows are one
 *   video (dataloader.py:107-116).  num_preds = 1 gives the training-mode output. */
int x3d_softmax_viewmean_fwd(const float* logits, float* probs, int N, int ncls, int num_preds,
                             void* stream);

/* ---- Row gather of the strided shortcut conv: ResBlock.residual, model.py:360-367 ------------
 * The 1x1x1 'valid' conv with stride (1,s,s) reads input pixels (t, ho*s, wo*s) only.  This
 * copies them into a dense matrix  out[(nt*Ho+ho)*Wo+wo, 0:C] = in[nt, ho*s, wo*s, 0:C]
 * (Ho=(Hi-1)/s+1, Wo=(Wi-1)/s+1, NT = N*T) that x3d_pw_tc_fwd then multiplies by the kernel. */
int x3d_gather_rows_fwd(const void* in, void* out, int NT, int Hi, int Wi, int stride, int C,
                        int dtype, void* stream);

/* ---- Head fully-connected layers: fc1 (+ReLU) and fc2 (+bias), model.py:119-121 -------------
 * (dropout, model.py:120, is the identity at inference.)  Small-M fp32 GEMM that streams the
 * weights once:  D[M, Nc] = act(A[M, K] . Wt[K, Nc] + bias),  act = ReLU if relu. */
int x3d_head_fc_fwd(const float* A, const float* Wt, const float* bias, float* D, int M, int K,
                    int Nc, int lda, int ldw, int ldd, int relu, void* stream);

/* ---- Pointwise convolution on the 5th-gen tensor cores (bf16 in, fp32 accumulate in TMEM) ----
 * Same contract as x3d_pw_fwd for a_dtype = d_dtype = X3D_BF16 and gather == 0, but the weights
 * are pre-packed bf16: Wp [Npad, Kpad] (K contiguous), Npad % 16 == 0, Kpad % 64 == 0, zero
 * padded, BN scale folded.  A tiles arrive by TMA (128B swizzle), tcgen05.mma accumulates in
 * TMEM, the epilogue adds bias (+ residual), applies ReLU and stores bf16.
 *
 * Second source (A2 != NULL; ResBlock's shortcut conv + bn_r folded into the projection conv,
 * model.py:360-367,386-392):  D = act(bias + pro(A) . W[0:K] + A2s . W[K1:K1+K2]) with
 *   A2   [a2_nt, a2_hi, a2_wi, K2] bf16 NDHWC block input (frames flattened), A2s[m] = A2[nt, s*ho, s*wo]
 *        for output pixel m = (nt*Ho + ho)*Wo + wo, Ho=(a2_hi-1)/s+1, Wo=(a2_wi-1)/s+1, s = a2_stride
 *        (the 'valid' stride-(1,s,s) 1x1x1 conv of the reference); M must equal a2_nt*Ho*Wo;
 *   Wp   holds the second source's K2 rows at packed column K1 = 64*ceil(K/64) (Kpad >= K1 + 64*ceil(K2/64));
 *   the prologue (se / swish) applies to the first source only; R must be NULL; bias = sum of both shifts.
 * Needs 128-pixel tiles that are whole rows of a frame or whole frames: x3d_pw_tc_sampler_supported
 * (1 / 0); otherwise gather with x3d_gather_rows_fwd and pass the shortcut's result as R.
 *
 * Column means (colmean != NULL; conv_5 + pool_5, model.py:117-118): additionally
 *   colmean[2*i + h, 0:Nc] = (1/64) * sum of the bf16-rounded outputs of rows 128*i + 64*h .. +63 (rows >= M
 *   contribute 0), fp32 [2*ceil(M/128), Nc]; the mean over the 64-row groups of a clip is the clip's
 *   global average pool when the clip has a multiple of 64 rows.  store_d = 0 then skips writing D. */
typedef struct x3d_pw_tc_args {
  const void* A; const void* Wp; const float* bias; const void* R; const float* se; void* D;
  int64_t M; int32_t K, Nc, lda, ldr, ldd, Kpad, Npad;
  int64_t rows_per_clip;
  int32_t swish, relu;
  const void* A2; int64_t a2_nt; int32_t K2, a2_stride, a2_hi, a2_wi;
  float* colmean; int32_t store_d, reserved;
} x3d_pw_tc_args;
int x3d_pw_tc_fwd(const x3d_pw_tc_args* args, void* stream);
int x3d_pw_tc_sampler_supported(int Hi, int Wi, int stride);

/* ---- Fused expand + channelwise: Bottleneck.a + bn_a + ReLU + b + bn_b (+ se_pool sums), ----
 * ---- model.py:306-312, as one kernel (bf16 storage) ------------------------------------------
 * Same result as x3d_pw_tc_fwd(relu=1) followed by x3d_dw3x3x3_fwd, but the `inner`-wide tensor
 * between the two convolutions stays in shared memory / TMEM (it is rounded to bf16 there exactly
 * as the unfused path rounds it when it stores it).
 *   x    [N,T,H,W,Cin] bf16          block input, Cin = stored channels (multiple of 8)
 *   wa   bf16 [Npad, Kpad]           packed expand kernel as for x3d_pw_tc_fwd (BN scale folded)
 *   bias_a [C] fp32                  bn_a shift;   wb [27,C] fp32, bias_b [C] fp32 as for x3d_dw3x3x3_fwd
 *   out  [N,T,Ho,Wo,C] bf16          Ho=ceil(H/s), Wo=ceil(W/s);  C = stored inner channels
 *   se_partial [N, nblk, C] fp32 or NULL, nblk = x3d_expand_dw_partial_blocks(...)
 * Returns X3D_ERR_UNSUPPORTED when no tile plan fits (the caller then runs the two kernels). */
int x3d_expand_dw_partial_blocks(int T, int H, int W, int Cin, int C, int stride);
int x3d_expand_dw_fwd(const void* x, const void* wa, const float* bias_a, const float* wb,
                      const float* bias_b, void* out, float* se_partial, int N, int T, int H,
                      int W, int Cin, int C, int Kpad, int Npad, int stride, int pad_h, int pad_w,
                      void* stream);

/* Same layers (model.py:306-316), persistent warp-specialised form: one CTA per SM walks (clip,
 * spatial tile) work items; TMA producer / tcgen05 issuer / TMEM drain warps / stencil warps / TMA
 * store run decoupled through mbarrier rings.  The expand result is kept in fp32 on chip (it is
 * NOT rounded to bf16 between the two convolutions, so the result is at least as close to the
 * reference's fp32 arithmetic as the unfused pair's).  Arguments as x3d_expand_dw_fwd, plus
 *   act  1: swish applied to the output (blocks without SE, model.py:316; se_partial must be NULL)
 *   se_partial [N, nblk, C], nblk = x3d_expand_dw2_partial_blocks(...) (0: no tile plan fits). */
int x3d_expand_dw2_partial_blocks(int T, int H, int W, int Cin, int C, int stride);
int x3d_expand_dw2_fwd(const void* x, const void* wa, const float* bias_a, const float* wb,
                       const float* bias_b, void* out, float* se_partial, int N, int T, int H,
                       int W, int Cin, int C, int Kpad, int Npad, int stride, int pad_h, int pad_w,
                       int act, void* stream);

/* ==== Either side of the forward path (SURVEY.md section 8f) ==================================
 * Input stage: utils.normalize, utils.py:42-72 (called from dataloader.py on decoded frames):
 *   out[p,c] = ((in[p,c] / norm_value) - mean[c]) / std[c]   in fp32, the reference's operation order.
 * `mean` / `std` are HOST pointers to 3 floats (cfg.DATA.MEAN / cfg.DATA.STD), read at call time.
 * in [pixels,3] uint8 (4-byte aligned) -> out [pixels,3] fp32 or bf16 (16-byte aligned). */
int x3d_normalize_u8(const uint8_t* in, void* out, int64_t pixels, const float* mean,
                     const float* std, float norm_value, int dtype, void* stream);
/* Evaluation clips of one decoded, already resized video, on the device: temporal views
 * (transforms.py:48-65: frame ((view*T + t) * max(1, F/T)) mod F, the video looped as often as
 * needed) and uniform spatial crops (transforms.py:149-190, 216-222: centre, or left / centre / right
 * along the longer side, offsets ceil((dim - S) / 2)), in the clip order dataloader.py:107-116 hands
 * to the model:   video [F,H,W,3] uint8 -> out [crops*views, T, S, S, 3] uint8 (crop-major). */
int x3d_eval_views_u8(const uint8_t* video, uint8_t* out, int F, int H, int W, int T, int views,
                      int crops, int S, void* stream);
/* Clips of decoded videos of any resolution (transforms.py:112-147, 192-227): per clip a bilinear
 * short-side resize of every source frame to rh x rw (tf.image.resize bilinear = TF 2.4
 * ResizeBilinear with half_pixel_centers, fp32 with every operation rounded separately, then a
 * truncating cast to uint8), an S x S crop at (y0, x0) of the resized frame and, for flip = 1, a
 * left-right flip of the crop:
 *   out[n][t][y][x][c] = resized(frame n,t)[y0 + y][x0 + (flip ? S-1-x : x)][c]
 *   frames     packed uint8 frames [*, H, W, 3] of a ragged batch of videos (device);
 *   frame_off  int64 [N*T] (device): byte offset in `frames` of the source frame of output frame (n, t);
 *   desc       x3d_clip_desc [N] (device): the source extent H x W, resized extent rh x rw, crop
 *              origin and flip of clip n;
 *   out        [N, T, S, S, 3] uint8 (4-byte aligned).
 * The descriptors are device data and are NOT checked by the call; the caller guarantees, per clip:
 * H, W >= 1; S <= rh, S <= rw; 0 <= y0 <= rh - S; 0 <= x0 <= rw - S; flip in {0, 1}; every frame
 * frame_off[n*T+t] .. + H*W*3 inside `frames`.  S <= 2048.  One launch covers the whole batch, so
 * every video can have its own frame count and frame size.  x3d_eval_views_u8 is this kernel over a
 * plan passed by value (rh = H, rw = W: an identity resize, which is exact). */
typedef struct x3d_clip_desc { int32_t H, W, rh, rw, y0, x0, flip; } x3d_clip_desc;
int x3d_video_clips_u8(const uint8_t* frames, const int64_t* frame_off, const x3d_clip_desc* desc, int N,
                       int T, int S, uint8_t* out, void* stream);
/* ---- Baseline JPEG decoding of the frames of TFRecord videos ------------------------------------
 * The reference reads GZIP TFRecords of SequenceExamples whose frames are JPEG images and decodes them
 * with tf.io.decode_jpeg (dataloader.py:66-91, 150-174; eval.py --tfrecord, train.py --use_tfrecord).
 * These three stages reproduce libjpeg-turbo's decompressor in its default libjpeg-6b mode (what TF 2.4
 * and Pillow link) bit for bit, for baseline sequential Huffman, 8-bit, three components in one
 * interleaved scan, luma sampling 2x2 or 1x1, chroma 1x1, no restart interval (x3d_tf_b200/jpeg.py
 * parses the headers and rejects everything else on the host).  Every frame of a ragged batch is
 * decoded by one launch per stage.
 *
 * Motion-JPEG frames (x3d_tf_b200/avi.py) add luma sampling 2x1 (4:2:2) and restart intervals, whose
 * intervals x3d_jpeg_entropy_rst decodes in parallel.
 *
 * Per frame (component c = 0 luma, 1 Cb, 2 Cr; hs, vs = luma sampling, 1 for chroma; an MCU holds the
 * hs*vs luma blocks in row-major order, then Cb, then Cr: 2x2 = 4 + 2 blocks, 2x1 = 2 side by side + 2):
 *   mcux = ceil(W / (8*hs)), mcuy = ceil(H / (8*vs));  component c has a block grid of
 *   bw_c x bh_c = (mcux*hs_c) x (mcuy*vs_c) blocks, stored component after component, each row-major:
 *   coefficients  int16 [blocks][64], natural order, quantised;  block b of the frame at
 *                 coef + (coef_off + b) * 64.  blocks = sum_c bw_c * bh_c.
 *   planes        uint8, plane c = [bh_c*8][bw_c*8] samples at plane_off + sum_{c'<c} bw_c'*bh_c'*64.
 *   output        packed row-major [H][W][3] RGB at out_off (4-byte aligned): exactly what
 *                 x3d_video_clips_u8 reads through frame_off.
 * The descriptors are device data and are NOT checked by the calls; the caller guarantees per frame:
 * 1 <= H, W <= 65535; (hs, vs) = (1, 1), (2, 2) or (2, 1); 0 <= tables < the number of table sets; the segment
 * seg_off .. + seg_len inside `data`; every buffer range above inside its buffer; status < the length
 * of `status`.  Ranges of different frames may not overlap. */
typedef struct x3d_jpeg_frame {
  int64_t seg_off;     /* byte offset in `data` of the entropy-coded segment (byte stuffing included) */
  int64_t coef_off;    /* first coefficient block */
  int64_t plane_off;   /* first byte of the sample planes */
  int64_t out_off;     /* first byte of the RGB output (multiple of 4) */
  int32_t seg_len;     /* bytes of the segment, up to (not including) the marker that ends it */
  int32_t H, W;
  int32_t hs, vs;      /* luma sampling factors */
  int32_t tables;      /* index of its x3d_jpeg_tables */
  int32_t status;      /* index of its status word */
  int32_t reserved;
} x3d_jpeg_frame;
/* One Huffman table as libjpeg's jpeg_make_d_derived_tbl derives it (jdhuff.c):
 *   maxcode[l]   largest code of length l (1..16), -1 if none; maxcode[17] = 0xFFFFF
 *   valoffset[l] huffval index of the first code of length l minus that code
 *   lookup[b]    for the next 8 bits b: (length << 8) | symbol of the code they start with, or 9 << 8
 *                when that code is longer than 8 bits */
typedef struct x3d_jpeg_huff {
  int32_t maxcode[18];
  int32_t valoffset[18];
  uint16_t lookup[256];
  uint8_t huffval[256];
} x3d_jpeg_huff;
/* The tables of one header (frames of one encoder run share it): quantisation tables in natural order
 * by table id, the derived DC / AC Huffman tables by table id, and which of them each component uses. */
typedef struct x3d_jpeg_tables {
  x3d_jpeg_huff dc[2];
  x3d_jpeg_huff ac[2];
  uint16_t q[4][64];
  int32_t comp_q[3], comp_dc[3], comp_ac[3];
  int32_t reserved;
} x3d_jpeg_tables;
enum x3d_jpeg_status {
  X3D_JPEG_OK = 0,
  X3D_JPEG_BAD_CODE = 1,       /* no Huffman code of length <= 16 matches */
  X3D_JPEG_BAD_RUN = 2,        /* a run of zeros or a coefficient past coefficient 63 */
  X3D_JPEG_SHORT_DATA = 3      /* the segment ended before the last block (libjpeg reads zeros there) */
};
enum x3d_jpeg_dct { X3D_JPEG_ISLOW = 0, X3D_JPEG_IFAST = 1 };
/* Stage 1, Huffman decoding (jdhuff.c decode_mcu): one warp per frame.  Writes every coefficient block
 * of the frame (zeros where no coefficient is coded) and status[frame.status] (x3d_jpeg_status); after
 * an error the remaining blocks of that frame are left as they were.  Never reads outside the frame's
 * segment or writes outside its blocks. */
int x3d_jpeg_entropy(const uint8_t* data, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                     int nframes, int16_t* coef, int32_t* status, void* stream);
/* Stage 1 for frames with a restart interval (DRI != 0): every interval is an independent bit stream whose
 * DC predictors start at 0, so one launch decodes all intervals of a ragged batch in parallel (one thread
 * per interval, each with its own bit reader that drops the stuffed 00 after every FF).  An interval
 * covers MCUs mcu0 .. mcu0 + nmcu - 1 of its frame in raster order; its bytes are data[off .. off + len)
 * (byte stuffing included, fill bytes and the RSTn / EOI marker that ends it excluded).  Writes every
 * block of those MCUs into the layout x3d_jpeg_entropy writes (zeros where no coefficient is coded).
 * An interval that fails raises its frame's status word to its x3d_jpeg_status with atomicMax (so the
 * result does not depend on the order of the intervals) and leaves its remaining blocks as they were:
 * the status words of the frames concerned must be zero before the launch.  Never reads outside an
 * interval or writes outside that interval's blocks.  The host (x3d_tf_b200/jpeg.py parse(mjpeg=True))
 * guarantees per interval: frame < the number of frames, mcu0 + nmcu <= the frame's MCU count, the byte
 * range inside `data`; the intervals of a frame cover each of its MCUs once. */
typedef struct x3d_jpeg_interval {
  int64_t off;         /* byte offset in `data` */
  int32_t len;         /* bytes */
  int32_t frame;       /* index of its x3d_jpeg_frame */
  int32_t mcu0;        /* first MCU (raster order) */
  int32_t nmcu;        /* MCUs */
} x3d_jpeg_interval;
int x3d_jpeg_entropy_rst(const uint8_t* data, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                         const x3d_jpeg_interval* intervals, int nintervals, int16_t* coef, int32_t* status,
                         void* stream);
/* Stage 2, dequantisation and 8x8 inverse DCT into the planes: method X3D_JPEG_ISLOW = jidctint.c
 * jpeg_idct_islow, X3D_JPEG_IFAST = jidctfst.c jpeg_idct_ifast with jddctmgr.c's multiplier table
 * (q * aanscales, descaled by 12 with rounding); both with IDCT_range_limit (wrap-around at RANGE_MASK).
 * max_blocks >= the block count of every frame. */
int x3d_jpeg_idct(const int16_t* coef, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                  int nframes, int max_blocks, int method, uint8_t* planes, void* stream);
/* Stage 3, upsampling and colour conversion into the output: chroma of 2x2 frames by jdsample.c
 * h2v2_fancy_upsample (edges replicated at the downsampled extent ceil(W/2) x ceil(H/2); the box
 * h2v2_upsample when ceil(W/2) <= 2, as libjpeg does), chroma of 2x1 frames by h2v1_fancy_upsample
 * (edges replicated at ceil(W/2); the box h2v1_upsample when ceil(W/2) <= 2), then jdcolor.c
 * ycc_rgb_convert.
 * max_pixels >= H*W of every frame. */
int x3d_jpeg_color(const uint8_t* planes, const x3d_jpeg_frame* frames, int nframes, int64_t max_pixels,
                   uint8_t* out, void* stream);
/* ---- Baseline JPEG encoding of video frames --------------------------------------------------------
 * Replaces the reference's tf.io.encode_jpeg(frame, quality=90) of every frame
 * (datasets/create_tfrecords.py:48-83).  These four stages reproduce libjpeg-turbo's compressor with
 * TF's settings bit for bit: JDCT_ISLOW, jpeg_set_quality(q, force_baseline = TRUE), the standard
 * (Annex K) Huffman tables or any others given in x3d_jpeg_enc_tables, no restart interval, three
 * components, luma sampling 2x2 (4:2:0) or 1x1 (4:4:4).  Each stage covers a ragged batch in one call
 * (one launch; two for the stuffing stage).
 * The host writes the headers (x3d_tf_b200/jpeg.py encoder_header) and appends EOI.
 *
 * Input: packed row-major [H][W][3] RGB uint8 frames at in_off in `rgb` (the layout x3d_jpeg_color
 * writes and x3d_video_clips_u8 reads).  Coefficients use the decoder's layout (above): component
 * after component, mcux*hs x mcuy*vs luma blocks then mcux x mcuy blocks of Cb and of Cr, int16 natural
 * order, block b at coef + (coef_off + b) * 64.  A frame's bit stream is MSB first in 32-bit words at
 * word_off in `words` (bit 0 = bit 31 of the first word); its entropy-coded segment (byte stuffing
 * included, padded with 1-bits) lands in `out` at the result's out_off.
 * The descriptors are device data and are NOT checked by the calls; the caller guarantees per frame:
 * 1 <= H, W <= 65535; hs = vs in {1, 2}; 0 <= tables < the number of table sets; the input frame, the
 * coefficient blocks, boff[coef_off .. + blocks) and words[word_off .. + word_cap) inside their
 * buffers; ranges of different frames do not overlap.  word_cap >= blocks * 52 + 1 always suffices
 * (a block codes to at most 1660 bits); a frame that needs more gets X3D_JPEG_OVERFLOW. */
typedef struct x3d_jpeg_enc_frame {
  int64_t in_off;      /* first byte of the RGB frame */
  int64_t coef_off;    /* first coefficient block, and first entry of boff */
  int64_t word_off;    /* first 32-bit word of the bit stream */
  int64_t word_cap;    /* words available there */
  int32_t H, W;
  int32_t hs, vs;      /* luma sampling factors: (2, 2) or (1, 1) */
  int32_t tables;      /* index of its x3d_jpeg_enc_tables */
  int32_t reserved;
} x3d_jpeg_enc_frame;
/* Quantisation tables (natural order: luma, chroma) and Huffman codes by symbol (jchuff.c
 * jpeg_make_c_derived_tbl ehufco / ehufsi) of DC luma, AC luma, DC chroma, AC chroma. */
typedef struct x3d_jpeg_enc_tables {
  uint16_t q[2][64];
  uint16_t code[4][256];
  uint8_t size[4][256];
} x3d_jpeg_enc_tables;
/* Per frame: bits of the entropy-coded data before padding (x3d_jpeg_enc_bits), the start of its
 * region in `out` (x3d_jpeg_enc_stuff, every frame), the length of its segment with byte stuffing, and
 * X3D_JPEG_OK or X3D_JPEG_OVERFLOW (word_cap or out_cap too small: then len is not written and
 * nothing of the frame is written to `words` or `out`). */
typedef struct x3d_jpeg_enc_result {
  int64_t bits;
  int64_t out_off;
  int64_t len;
  int32_t status;
  int32_t reserved;
} x3d_jpeg_enc_result;
#define X3D_JPEG_OVERFLOW 4
/* Stage A: jccolor.c rgb_ycc_convert (16-bit fixed point), the last column and row replicated
 * (jcsample.c expand_right_edge, jcprepct.c expand_bottom_edge), chroma of 4:2:0 by jcsample.c
 * h2v2_downsample (bias 1, 2) with its last row replicated to the MCU height, jfdctint.c
 * jpeg_fdct_islow and jcdctmgr.c's quantisation by reciprocal (compute_reciprocal of q << 3 with
 * libjpeg-turbo's 16-bit DCTELEM).  The luma blocks of 4:2:0 frames past ceil(W/8) x ceil(H/8) are
 * jccoefct.c's dummy blocks: AC zero, DC that of the block before them in the MCU.
 * max_blocks >= the block count of every frame. */
int x3d_jpeg_fdct(const uint8_t* rgb, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                  int nframes, int max_blocks, int16_t* coef, void* stream);
/* Stage B: the code length of every block (jchuff.c encode_one_block: DC difference to the previous
 * block of the component in scan order, AC run lengths with ZRL and EOB), an exclusive scan per frame
 * into boff[coef_off + scan position] (int64 bit offsets), res[f].bits and res[f].status, and zeroes
 * the frame's ceil(bits / 32) words.  One CTA per frame. */
int x3d_jpeg_enc_bits(const int16_t* coef, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                      int nframes, int64_t* boff, x3d_jpeg_enc_result* res, uint32_t* words, void* stream);
/* Stage C1: every block's codes ORed into the frame's words at its bit offset; the last block pads the
 * stream to a byte with 1-bits (jchuff.c flush_bits).  Frames whose status is not X3D_JPEG_OK are
 * skipped.  max_blocks as for x3d_jpeg_fdct. */
int x3d_jpeg_enc_emit(const int16_t* coef, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                      int nframes, int max_blocks, const int64_t* boff, const x3d_jpeg_enc_result* res,
                      uint32_t* words, void* stream);
/* Stage C2: byte stuffing (0x00 after every 0xFF) into `out` (out_cap bytes).  A first launch (one CTA)
 * writes res[f].out_off for every frame: the sum over frames f' < f of 2 * ceil(bits_f' / 8), a bound
 * of their stuffed lengths, so out_cap >= 2 * the sum over all frames suffices.  The second (one CTA per
 * frame) stuffs every X3D_JPEG_OK frame whose region fits and writes res[f].len; a frame whose region
 * ends past out_cap gets X3D_JPEG_OVERFLOW. */
int x3d_jpeg_enc_stuff(const uint32_t* words, const x3d_jpeg_enc_frame* frames, int nframes,
                       x3d_jpeg_enc_result* res, uint8_t* out, int64_t out_cap, void* stream);

/* x3d_stem_tc_fwd with the input stage fused into its loader: uint8 NDHWC clips in, bf16
 * activations out (same result as x3d_normalize_u8(bf16) followed by x3d_stem_tc_fwd). */
int x3d_stem_tc_u8_fwd(const uint8_t* in, const float* mean, const float* std, float norm_value,
                       const void* wc, const float* bias, void* out, int N, int T, int H, int W,
                       int C, int kt, void* stream);
/* Evaluation metrics, eval.py:62-70 (model.compile(loss=SparseCategoricalCrossentropy, metrics=
 * [SparseCategoricalAccuracy, SparseTopKCategoricalAccuracy(k=5)])):  probs [V,ncls] fp32, labels
 * [V] int32;  acc[0] += sum of losses, acc[1] += top-1 hits, acc[2] += top-k hits, acc[3] += V
 * (caller-zeroed fp64[4] on the device, so shards and batches accumulate). */
int x3d_eval_metrics(const float* probs, const int32_t* labels, double* acc, int V, int ncls,
                     int k, void* stream);

/* ==== Training step (BASELINE configs[4]; train.py:85-152 -> Keras train_step) ================
 * fp32, channels-last, activations viewed as [M, C] matrices (M = N*T*H*W).  Reductions accumulate
 * into caller-zeroed fp64 buffers.  The forward convolutions of the training step are the entry
 * points above called with raw (un-folded) kernels and no bias; what follows is everything else. */

/* Per-channel reductions over rows, one result pair per segment of `seg_rows` rows:
 *   mode 0: out[s][0][c] += sum a,  out[s][1][c] += sum a^2         (BatchNorm batch statistics)
 *   mode 1: out[s][0][c] += sum g,  out[s][1][c] += sum g*xhat      (BatchNorm backward;
 *           g = a masked by relu_out > 0 if relu_out != NULL, xhat = (x - mean) * rstd)
 *   mode 2: out[s][0][c] += sum a                                    (bias gradients, SE pooling) */
int x3d_colreduce(const float* a, const float* x, const float* mean, const float* rstd,
                  const float* relu_out, int64_t M, int C, int64_t seg_rows, double* out, int mode,
                  void* stream);
/* BatchNormalization(training=True), model.py:89,196,254,268,300,368: batch mean / biased variance
 * from the mode-0 sums, rstd = 1/sqrt(var+eps); moving = momentum*moving + (1-momentum)*batch. */
int x3d_bn_finalize(const double* sums, int64_t M, int C, float eps, float momentum, float* mean,
                    float* var, float* rstd, float* mov_mean, float* mov_var, void* stream);
int x3d_bn_apply_fwd(const float* x, const float* mean, const float* rstd, const float* gamma,
                     const float* beta, float* y, int64_t M, int C, int relu, void* stream);
/* dx = gamma*rstd*(g - sum_g/M - xhat*sum_gxhat/M) with the mode-1 sums (which are also dbeta, dgamma) */
int x3d_bn_bwd_apply(const float* dy, const float* x, const float* relu_out, const float* mean,
                     const float* rstd, const float* gamma, const double* sums, float* dx, int64_t M,
                     int C, void* stream);
int x3d_d2f(const double* in, float* out, int64_t n, float scale, void* stream);
/* Backward-filter of a 1x1x1 conv (a, c, residual, conv5, fc1, fc2, se_fc1, se_fc2):
 * dW[k,n] += sum_m A[row(m),k] * dD[m,n]; gather/geometry as in x3d_pw_fwd.  (Backward-data is
 * x3d_pw_fwd with the transposed kernel.)  3xTF32 tensor-core path when K, N, lda, ldd are multiples
 * of 4 and the pointers 16-byte aligned (fp32 partial sums per 32-row chunk), CUDA cores otherwise;
 * fp64 atomics into dW either way. */
int x3d_pw_wgrad(const float* A, const float* dD, double* dW, int64_t M, int K, int N, int lda,
                 int ldd, int gather, int Ho, int Wo, int Hi, int Wi, int stride, void* stream);
/* The backward-filter of the mixed-precision step: dW[k,n] += sum_m bf16(A[row(m),k]) * bf16(dD[m,n])
 * (round-to-nearest-even), mma.sync m16n8k16 bf16 with fp32 partial sums per 32-row chunk, fp64 atomics
 * into dW.  Arguments as x3d_pw_wgrad; K, N, lda, ldd multiples of 4, A and dD 16-byte aligned. */
int x3d_pw_wgrad_bf16(const float* A, const float* dD, double* dW, int64_t M, int K, int N, int lda,
                      int ldd, int gather, int Ho, int Wo, int Hi, int Wi, int stride, void* stream);
/* Backward-data / backward-filter of the channelwise 3x3x3 conv (Bottleneck.b, model.py:259-267) */
int x3d_dw_dgrad(const float* dy, const float* w, float* dx, int N, int T, int H, int W, int C,
                 int stride, int pad_h, int pad_w, void* stream);
int x3d_dw_wgrad(const float* x, const float* dy, double* dwt, int N, int T, int H, int W, int C,
                 int stride, int pad_h, int pad_w, void* stream);
/* Stem in training form (model.py:202-208): conv_s and conv_t as separate ops so that the conv_s
 * output can be kept for conv_t's backward-filter; flip=1 turns x3d_tconv_fwd into backward-data. */
int x3d_stem_convs_fwd(const float* in, const float* ws, float* out, int N, int T, int H, int W,
                       int C, void* stream);
int x3d_stem_convs_wgrad(const float* in, const float* ds, double* dws, int N, int T, int H, int W,
                         int C, void* stream);
int x3d_tconv_fwd(const float* in, const float* wt, float* out, int N, int T, int64_t P, int C,
                  int kt, int flip, void* stream);
int x3d_tconv_wgrad(const float* s, const float* dy, double* dwt, int N, int T, int64_t P, int C,
                    int kt, void* stream);
/* out = swish(y * s[clip,c]) and its backward (dy, ds[clip,c] += sum dv*y), model.py:311-316 */
int x3d_scale_swish_fwd(const float* y, const float* s, float* out, int64_t M, int C,
                        int64_t rows_per_clip, void* stream);
int x3d_scale_swish_bwd(const float* dout, const float* y, const float* s, float* dy, double* ds,
                        int64_t M, int C, int64_t rows_per_clip, void* stream);
/* Elementwise: op 0 relu(a+b) | 1 a*(b>0) | 2 sigmoid(a) | 3 a*b*(1-b) | 4 a+b | 5 a*b */
int x3d_ew(const float* a, const float* b, float* out, int64_t n, int op, void* stream);
/* Backward of the global average pool (AdaptiveAvgPool3D, model.py:473-483) */
int x3d_pool_bwd(const float* dm, float* dy, int64_t M, int C, int64_t rows_per_clip, float scale,
                 int accumulate, void* stream);
/* Backward-data of the strided shortcut conv: dst[nt, ho*s, wo*s, :] += src[nt, ho, wo, :] */
int x3d_strided_add(const float* src, float* dst, int NT, int Ho, int Wo, int Hi, int Wi,
                    int stride, int C, void* stream);
int x3d_dropout_mask(float* mask, int64_t n, float rate, uint64_t seed, void* stream);
/* Softmax + SparseCategoricalCrossentropy on probabilities (train.py:104) and d loss / d logits * gscale */
int x3d_softmax_xent(const float* logits, const int32_t* labels, float* loss, float* dlogits, int N,
                     int ncls, float gscale, void* stream);
/* SGD(nesterov=True) + L2, train.py:88-92, model.py:47:  g = grad + wd*w; v = mu*v - lr*g; w += mu*v - lr*g */
int x3d_sgd_nesterov_step(float* w, const float* grad, float* v, const float* wd, int64_t n,
                          float lr, float momentum, void* stream);
/* Adam, train.py:93-95 (Keras defaults):  g = grad + wd*w; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
 * w -= lr_t m / (sqrt(v) + eps), with lr_t = lr sqrt(1 - b2^t) / (1 - b1^t) passed by the caller. */
int x3d_adam_step(float* w, const float* grad, float* m, float* v, const float* wd, int64_t n,
                  float lr_t, float beta1, float beta2, float eps, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* X3D_B200_H_ */
