/*
 * msg_b200.h -- C-ABI of the B200-native (sm_100a) multi-style GAN hot path.
 *
 * The reference (regicide211212/multi-style-transfer-gan) is 100 % Python and has no FFI layer
 * (SURVEY.md 2.1); its "operator interface" for this path is the set of torch.nn library ops its
 * modules dispatch.  Each entry point below names the reference call site (file:line, relative to
 * the reference root) whose library op it replaces.  The Python drop-in classes in
 * multi_style_transfer_gan_b200/ bind these with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain C: raw DEVICE pointers, explicit sizes, cudaStream_t passed as void*.
 *   - every function returns 0 on success or a negative MSG_ERR_* code; msg_last_error() gives a
 *     thread-local message.  No exceptions, no allocation, no ownership transfer: the caller owns
 *     inputs, outputs and workspaces.
 *   - activations are NHWC ("pixel-major, channel-contiguous"), dtype MSG_F32 or MSG_BF16; all
 *     statistics, gradients of parameters and optimizer state are fp32.
 *   - the library refuses to run on anything but compute capability 10.x (no fallback).
 */
#ifndef MSG_B200_H_
#define MSG_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSG_OK 0
#define MSG_ERR_SHAPE (-1)
#define MSG_ERR_ALIGN (-2)
#define MSG_ERR_ARCH (-3)
#define MSG_ERR_CUDA (-4)
#define MSG_ERR_UNSUPPORTED (-5)

#define MSG_F32 0
#define MSG_BF16 1

/* epilogue / elementwise activations */
#define MSG_ACT_NONE 0
#define MSG_ACT_RELU 1
#define MSG_ACT_LRELU 2 /* LeakyReLU(0.2), enhanced_generator.py:238 */
#define MSG_ACT_TANH 3  /* enhanced_generator.py:138 */

/* msg_conv_desc.flags */
#define MSG_CONV_STATS 1u      /* accumulate per-(n,cout) sum / sum-of-squares of the output   */
#define MSG_CONV_OUT_NCHW_F32 2u /* write the result as fp32 NCHW (final image, Cout small)     */
#define MSG_CONV_ACCUM 8u      /* y += result (sums the gradient branches of a fan-out)          */
#define MSG_CONV_PER_IMAGE_W 16u /* w holds one packed weight per image, [N][Cout][KH*KW*Cin]: a batched
                                   * "matrix times per-image matrix" (Gram backward).  bf16 TMA kernel only.    */
#define MSG_CONV_FORCE_GATHER 512u /* debugging: skip the TMA kernel, use the cp.async gather kernel  */
#define MSG_CONV_FORCE_SIMT 256u /* debugging: never take the tcgen05 path                      */
#define MSG_CONV_IN_NORM 4u    /* normalise the INPUT on load with in_stats (IN + act fused
                                   into the consumer's operand fetch)                             */

/* weight packing modes for msg_pack_conv_weight */
#define MSG_PACK_FWD 0        /* OIHW            -> [O][KH][KW][I]                                */
#define MSG_PACK_DGRAD_S1 1   /* OIHW            -> [I][KH-1-kh][KW-1-kw][O]  (stride-1 dgrad)    */
#define MSG_PACK_CONVT_PHASES 2 /* [I][O][4][4]  -> [4 phases][O][2][2][I]    (4x4 s2 p1 convT)   */

const char* msg_last_error(void);
int msg_version(void);
/* 0 if the current device is sm_100 (B200); MSG_ERR_ARCH otherwise. */
int msg_check_device(void);
int msg_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * Generic "gather convolution" (implicit GEMM).  One descriptor covers every conv on the path:
 *   Conv2d 7x7 s1 p3 (enhanced_generator.py:92,137), Conv2d 4x4 s2 p1 (:99,106,237-249),
 *   the 1x1 qkv/proj/branch1/fusion convs (:10,11,53,73), the dilated 3x3 branches (:58,63,68),
 *   each sub-pixel phase of ConvTranspose2d 4x4 s2 p1 (:121,128), D heads (:256,262,265),
 *   and, with re-packed weights, every dgrad of the above.
 *
 *   for (n, i, j) in [N, Hg, Wg], co in [0, Cout):
 *     acc = bias[co] + sum_{th<KH, tw<KW, ci<Cin}
 *             x[n, i*in_stride - pad_h + th*dil, j*in_stride - pad_w + tw*dil, ci_off + ci]   (0 outside)
 *             * w[co][th][tw][ci]
 *     y[n, i*out_stride + out_off_h, j*out_stride + out_off_w, co_off + co] = act(acc)
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int dtype;                            /* MSG_F32 / MSG_BF16: x, w, y                          */
  int N;
  int Hi, Wi, Ci_total, ci_off, Cin;    /* input tensor [N,Hi,Wi,Ci_total], channel slice used  */
  int Ho, Wo, Co_total, co_off, Cout;   /* output tensor [N,Ho,Wo,Co_total], slice written      */
  int Hg, Wg;                           /* GEMM pixel grid                                      */
  int KH, KW, in_stride, pad_h, pad_w, dil;
  int out_stride, out_off_h, out_off_w;
  int act;                              /* MSG_ACT_*                                            */
  unsigned flags;                       /* MSG_CONV_*                                           */
  int in_act;                           /* activation applied after the fused input norm        */
} msg_conv_desc;

/* x, w (packed [Cout][KH*KW*Cin], dtype), bias fp32 [Cout] or NULL, y, stats fp64 [N][Co_total][2]
 * (only with MSG_CONV_STATS; must be zeroed by the caller; accumulates across calls),
 * in_stats fp64 [N][Ci_total][2] raw sums of the input plane (only with MSG_CONV_IN_NORM). */
int msg_conv2d(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
               double* stats, const double* in_stats, void* stream);
/* Which engine msg_conv2d would take for this descriptor / these pointers, without launching anything:
 * 2 = persistent TMA + tcgen05 kernel, 1 = cp.async gather + tcgen05 kernel, 0 = SIMT engine, < 0 = MSG_ERR_*.
 * (Callers use it to decide whether fusing the input InstanceNorm into a 1x1 conv is profitable.) */
int msg_conv2d_path(const msg_conv_desc* d, const void* x, const void* w, const void* y);

/* ---------------------------------------------------------------------------------------------
 * InstanceNorm affine of a style-conditional generator.  Every site that applies an InstanceNorm
 * (the stand-alone apply, and the convs / stages below that normalise their input on load) can
 * take an optional affine, passed as (gamma, beta, img_stride), fp32:
 *   gamma[n * img_stride + c] is indexed exactly like the statistics it accompanies (channel
 *   offsets ci_off / cs_off included); img_stride 0 is one [C] affine for the whole batch;
 *   gamma = beta = NULL is no affine (the entry points without the _affine suffix pass NULL).
 * The apply is z = fmaf(x, scale, shift), scale = rstd * gamma[..], shift = beta[..] - mean * scale,
 * so gamma = 1, beta = 0 gives the affine-free result bit for bit.
 * ------------------------------------------------------------------------------------------- */
/* msg_conv2d with an input affine for MSG_CONV_IN_NORM.  Only the TMA + tcgen05 kernel applies one
 * (msg_conv2d_path == 2): a descriptor that would run on another engine returns MSG_ERR_SHAPE. */
int msg_conv2d_affine(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y, double* stats,
                      const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride, void* stream);
/* Per-image affine tables of all the normalisation sites of a forward in one launch:
 *   gamma_out[n][c] = sum_s w[n][s] * gammas[s][c]  (beta alike), c < Ct,
 * an fmaf chain over s in ascending order starting from 0 -- the chain msg_instnorm_apply runs
 * over its w[S], so a row equals that apply's blended affine bit for bit.
 * w fp32 [N][S] (weights used as given, no normalisation); gammas, betas fp32 [S][Ct];
 * gamma_out, beta_out fp32 [N][Ct]. */
int msg_style_affine(const float* w, int N, int S, const float* gammas, const float* betas, int Ct, float* gamma_out,
                     float* beta_out, void* stream);
/* Backward of msg_style_affine for one sums arena [N][Ct][2] fp64 (the per-(image, channel)
 * (sum g, sum g * xhat) = (d beta_n, d gamma_n) of msg_instnorm_bwd_reduce_affine):
 *   dgammas[s][c] += sum_n w[n][s] * sums[n][c][1],  dbetas[s][c] += sum_n w[n][s] * sums[n][c][0]
 * (fp64 sum over n in ascending order, one fp32 add).  dgammas, dbetas fp32 [S][Ct]. */
int msg_style_affine_bwd(const double* sums, const float* w, int N, int S, int Ct, float* dgammas, float* dbetas,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * "Row-slab" convolution (bf16, W % 8 == 0): stride-1, same-size convs with small N, several taps
 * sharing one input row slab -- the 7x7 convs (enhanced_generator.py:92,137) and the fused
 * MultiScaleBlock branches (:52-71, one launch writes the concatenated tensor).  A k-block is an
 * (input row offset dy, 64-channel block cb) pair; each of its taps has a horizontal shift sx, its
 * own [ncols x 64] weight tile (row tp*ncols of w_slab) and an accumulator column offset.
 *   acc[x][tap_acc_col[tp] + c] (+)= sum_k x[n, y + kb_dy, x + tap_sx[tp], cb*64 + k] * w_slab[tp*ncols + c][k]
 * pixel_pair_k (3-channel image padded to 8 channels): K=16 of one MMA = this pixel and the next;
 * all taps of a k-block share w_slab tile kb, tap_kstep selects the 16-wide K slice.
 * ------------------------------------------------------------------------------------------- */
#define MSG_SLAB_MAX_KBLOCKS 32
#define MSG_SLAB_MAX_TAPS 128
typedef struct {
  int dtype;
  int N, H, W, Ci_total, ci_off, Cin;
  int Co_total, co_off;
  int out_stride;  /* 0 / 1: y is [N,H,W,Co_total].  2: output pixel (y, x) of the conv lands at row
                      2y + out_off_h, column 2x + out_off_w of y [N,2H,2W,Co_total]: one sub-pixel phase
                      of a 4x4 stride-2 transposed conv run as a 2x2 conv on its row slabs
                      (enhanced_generator.py:120-121, 127-128).  bf16 NHWC output only.              */
  int out_off_h, out_off_w;
  int Ntot;        /* accumulator columns (multiple of 16, <= 256)                                */
  int n_store;     /* leading columns actually written to y (<= Ntot)                             */
  int ncols;       /* columns per tap (multiple of 16)                                            */
  int halo;        /* max |tap_sx|                                                                */
  int pixel_pair_k;
  int n_chains;    /* 1, 2 or 4 independent accumulation chains (TMEM column groups Ntot apart, summed
                      in the epilogue): back-to-back tcgen05.mma into the SAME columns are latency-bound
                      when N is small; n_chains * Ntot <= 256                                       */
  int act;
  unsigned flags;  /* MSG_CONV_STATS | MSG_CONV_OUT_NCHW_F32                                      */
  int n_kblocks, n_taps;
  int kb_dy[MSG_SLAB_MAX_KBLOCKS], kb_cb[MSG_SLAB_MAX_KBLOCKS], kb_tap_begin[MSG_SLAB_MAX_KBLOCKS + 1];
  int tap_sx[MSG_SLAB_MAX_TAPS], tap_acc_col[MSG_SLAB_MAX_TAPS], tap_first[MSG_SLAB_MAX_TAPS],
      tap_kstep[MSG_SLAB_MAX_TAPS];
} msg_slab_desc;
/* x [N,H,W,Ci_total] bf16; w_slab bf16 [n_tiles*ncols][64]; bias fp32 [Ntot] or NULL (program column
 * order); y [N,H,W,Co_total] bf16 (or fp32 NCHW [N,Co_total,H,W] with MSG_CONV_OUT_NCHW_F32);
 * stats fp64 [N][Co_total][2] accumulated (MSG_CONV_STATS). */
int msg_conv_slab(const msg_slab_desc* d, const void* x, const void* w_slab, const float* bias, void* y,
                  double* stats, void* stream);

/* ---------------------------------------------------------------------------------------------
 * "Taps-as-N" row-slab convolution (bf16, Cin % 64 == 0): all filter taps sharing an input row are ONE
 * MMA (filters stacked along N over the unshifted slab); the horizontal shifts are applied in the
 * epilogue.  Used for the 7x7 output conv (enhanced_generator.py:137) and the fused MultiScaleBlock
 * branches at C = 64 (:52-71).  k-block kb: slab row y + kb_dy, channel block kb_cb, weight rows
 * [kb_wrow, kb_wrow + kb_ncols) of w_rows ([rows][64] bf16) -> accumulator columns [kb_col0, +kb_ncols).
 * Output group g:  out[x][grp_out_col0 + c] = sum_{terms} acc[x + term_shift][grp_col0 + term_col + c],
 * c < grp_out_cols (<= 16), x in [0, 128 - 2*halo).
 * ------------------------------------------------------------------------------------------- */
#define MSG_SHIFT_MAX_KBLOCKS 32
#define MSG_SHIFT_MAX_GROUPS 8
#define MSG_SHIFT_MAX_TERMS 32
typedef struct {
  int dtype;
  int N, H, W, Ci_total, ci_off, Cin;
  int Co_total, co_off;
  int Ntot;        /* accumulator columns (multiple of 16, <= 256)  */
  int n_out;       /* output columns (<= 64); bias / stats indexing */
  int halo;
  int act;
  unsigned flags;  /* MSG_CONV_STATS | MSG_CONV_OUT_NCHW_F32 */
  int n_kblocks, n_groups, n_terms;
  int kb_dy[MSG_SHIFT_MAX_KBLOCKS], kb_cb[MSG_SHIFT_MAX_KBLOCKS], kb_col0[MSG_SHIFT_MAX_KBLOCKS],
      kb_ncols[MSG_SHIFT_MAX_KBLOCKS], kb_wrow[MSG_SHIFT_MAX_KBLOCKS], kb_first[MSG_SHIFT_MAX_KBLOCKS];
  int grp_col0[MSG_SHIFT_MAX_GROUPS], grp_span[MSG_SHIFT_MAX_GROUPS], grp_out_col0[MSG_SHIFT_MAX_GROUPS],
      grp_out_cols[MSG_SHIFT_MAX_GROUPS], grp_term_begin[MSG_SHIFT_MAX_GROUPS + 1];
  int term_shift[MSG_SHIFT_MAX_TERMS], term_col[MSG_SHIFT_MAX_TERMS];
  /* Multi-row tiles (the kernel is bound by L2 -> SM slab bytes): a tile produces tile_rows (0 / 1: one) consecutive
   * output rows; k-block kb with kb_same_slab[kb] != 0 re-uses the slab of k-block kb-1 (same input row, another
   * output row's filter row, other accumulator columns); output group g belongs to output row y + grp_row[g].
   * 7x7 conv with tile_rows = 2: 8 slabs per 2 rows instead of 14. */
  int tile_rows;
  int kb_same_slab[MSG_SHIFT_MAX_KBLOCKS];
  int grp_row[MSG_SHIFT_MAX_GROUPS];
} msg_shift_desc;
int msg_conv_shift(const msg_shift_desc* d, const void* x, const void* w_rows, const float* bias, void* y,
                   double* stats, void* stream);

/* wgrad of the same descriptor: dw[co][th][tw][ci] (fp32, packed layout, ACCUMULATED into) =
 * sum over pixels of dy[..., co] * gathered x[..., ci].  Replaces autograd's conv weight grads for
 * every conv above (enhanced_train.py:84,121). */
int msg_conv2d_wgrad(const msg_conv_desc* d, const void* x, const void* dy, float* dw_packed,
                     void* stream);

/* fp32 master weight (PyTorch layout) -> packed operand of `dtype`.  O, I are the leading two dims
 * of the source tensor as stored by PyTorch (Conv2d: O=Cout, I=Cin; ConvTranspose2d: O=Cin, I=Cout
 * for MSG_PACK_CONVT_PHASES pass the tensor as stored, O=dim0, I=dim1).  `scale` (device fp32
 * scalar or NULL) multiplies by 1/(*scale): spectral norm's weight_orig / sigma
 * (enhanced_generator.py:269-271). */
int msg_pack_conv_weight(const float* w, int dim0, int dim1, int KH, int KW, int mode, int dtype,
                         const float* inv_scale_denominator, void* out, void* stream);
/* inverse scatter of a packed fp32 gradient back to PyTorch layout (accumulates: dst += src). */
int msg_unpack_conv_wgrad(const float* dw_packed, int dim0, int dim1, int KH, int KW, int mode,
                          float* dw, void* stream);

/* column sums: db[c] += sum over rows of dy[row][c_off + c]  (bias gradients). */
int msg_bias_grad(int dtype, const void* dy, long long rows, int C_total, int c_off, int C,
                  float* db, void* stream);

/* ---------------------------------------------------------------------------------------------
 * InstanceNorm2d(affine=False, eps=1e-5, biased variance) -- enhanced_generator.py:54,59,64,69,
 * 74,93,100,107,122,129,242,246,250,263.  Bandwidth-bound, vectorised, warp-shuffle reductions.
 * stats are RAW plane sums, fp64 [N][C][2] = (sum x, sum x^2) over H*W: fp64 makes
 * var = E[x^2] - mean^2 cancellation-free and the atomics order-independent (parity mode needs it).
 * ------------------------------------------------------------------------------------------- */
int msg_instnorm_stats(int dtype, const void* x, int N, long long HW, int C, double* stats,
                       void* stream);
/* y = act((x - mean) * rstd * gamma + beta) [+ residual];   gamma/beta optional blended affine:
 * gamma[c] = sum_s w[s]*gammas[s][c] (north_star extension; pass S=0 for the reference's
 * affine-free norm).  residual may be NULL.  y may alias x. */
int msg_instnorm_apply(int dtype, const void* x, const double* stats, int N, long long HW, int C,
                       int act, const void* residual, int S, const float* gammas,
                       const float* betas, const float* w, void* y, void* stream);
/* msg_instnorm_apply with an affine table (gamma, beta, img_stride) instead of the blend; S > 0
 * together with a table is refused.  msg_instnorm_apply is this with a NULL table. */
int msg_instnorm_apply_affine(int dtype, const void* x, const double* stats, int N, long long HW, int C, int act,
                              const void* residual, int S, const float* gammas, const float* betas, const float* w,
                              const float* gamma, const float* beta, int img_stride, void* y, void* stream);
/* backward of y = act(IN(x)) [+ residual]:  given dy, x (pre-norm) and stats, writes dx.
 * (d residual = dy is the caller's business.)  scratch: fp64 [N][C][2], zeroed by the callee. */
int msg_instnorm_bwd(int dtype, const void* x, const double* stats, const void* dy, int N,
                     long long HW, int C, int act, double* scratch, void* dx, void* stream);
/* The two halves of msg_instnorm_bwd, for a backward that runs a collective between them
 * (synchronised BatchNorm: sum the per-channel reductions over the ranks, then apply).
 * gamma, beta: optional per-channel affine, fp32 [C] (both NULL: none).  The forward was
 * y = act(z), z = fmaf(x, scale, shift), scale = rstd * gamma, shift = beta - mean * scale
 * (msg_instnorm_apply with S = 1, w = {1}); g = dy * act'(z) takes its mask from z rebuilt with
 * that same arithmetic, so it equals the sign of the stored y and y need not be read.
 *   reduce: zeroes sums, then sums[n][c] = (sum g, sum g * xhat) in fp64.
 *   apply:  dx = gamma * rstd * (g - sums[n][c][0] / HW - xhat * sums[n][c][1] / HW), rounded to
 *           the storage type once.
 * Statistics convention: every stats / sums a kernel sees is normalised to the LOCAL element
 * count HW.  A caller that reduces over M_global elements held on several ranks scales the
 * all-reduced global sums by HW_local / M_global (in fp64) before handing them to a kernel; with
 * one rank that factor is exactly 1, and msg_instnorm_apply serves the synchronised forward. */
int msg_instnorm_bwd_reduce(int dtype, const void* x, const double* stats, const void* dy, int N,
                            long long HW, int C, int act, const float* gamma, const float* beta,
                            double* sums, void* stream);
int msg_instnorm_bwd_apply(int dtype, const void* x, const double* stats, const void* dy, int N,
                           long long HW, int C, int act, const float* gamma, const float* beta,
                           const double* sums, void* dx, void* stream);
/* The same with a per-image affine (gamma, beta, img_stride): the reductions of image n are then
 * d beta_n and d gamma_n.  With img_stride > 0 the sums rows are img_stride apart as well
 * (sums [N][img_stride][2], the columns of this call written, the others untouched), so the calls
 * of one backward fill one arena laid out like the affine tables.  The functions above are these
 * with img_stride 0. */
int msg_instnorm_bwd_reduce_affine(int dtype, const void* x, const double* stats, const void* dy, int N, long long HW, int C,
                                   int act, const float* gamma, const float* beta, int img_stride, double* sums, void* stream);
int msg_instnorm_bwd_apply_affine(int dtype, const void* x, const double* stats, const void* dy, int N, long long HW, int C,
                                  int act, const float* gamma, const float* beta, int img_stride, const double* sums, void* dx,
                                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * LocalAttention core (enhanced_generator.py:22-35) on a [N,H,W,3C] qkv map (the 1x1 qkv conv is
 * msg_conv2d): per ws x ws window, L2-normalise q and k over C per pixel (eps 1e-12), C x C
 * logits, softmax over the last dim, times v.  out: [N,H,W,C].  No scale, no residual.
 * ------------------------------------------------------------------------------------------- */
int msg_local_attn_fwd(int dtype, const void* qkv, int N, int H, int W, int C, int ws, void* out,
                       void* stream);
int msg_local_attn_bwd(int dtype, const void* qkv, const void* dout, int N, int H, int W, int C,
                       int ws, void* dqkv, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused LocalAttention STAGE (the whole of LocalAttention.forward, enhanced_generator.py:13-47, window_size 4)
 * as ONE tcgen05 kernel: [optional InstanceNorm + ReLU of the producer, from its raw plane sums] -> qkv 1x1 conv
 * -> window attention (logits and probabilities never leave the SM: S in TMEM, P written back to TMEM and fed
 * to the P.V MMA from there) -> proj 1x1 conv.  Replaces msg_conv2d(qkv) + msg_local_attn_fwd + msg_conv2d(proj)
 * on the inference path; HBM traffic = x in + out.
 *   x      [N,H,W,C]  bf16 NHWC (raw conv output when in_stats != NULL, else the already normalised input)
 *   in_stats  fp64 [N][C][2] raw plane sums of x (msg_conv2d's MSG_CONV_STATS output) or NULL; in_act: MSG_ACT_NONE/RELU
 *   wqkv   [3C][C] bf16 (msg_pack_conv_weight MSG_PACK_FWD of qkv.weight), bqkv fp32 [3C]
 *   wproj  [C][C]  bf16 (same packing of proj.weight), bproj fp32 [C]
 *   out    [N,H,W,C]  bf16
 * Supported: bf16, C in {64, 128}, H % 4 == 0, W % 4 == 0, 16-byte aligned pointers (msg_la_stage_supported
 * returns 1); anything else: the three separate calls above.
 * ------------------------------------------------------------------------------------------- */
int msg_la_stage_supported(int dtype, int N, int H, int W, int C, const void* x, const void* wqkv,
                           const void* wproj, const void* out);
/* development hook, effective only in builds with -DMSG_LA_TRACE: device buffer (19 x 4096 u64) that receives the
 * role timelines of CTA 0 (tools/la_trace.py); NULL switches it off. */
int msg_la_stage_set_trace(void* buf);
int msg_la_stage_fwd(int dtype, const void* x, const double* in_stats, int in_act, const void* wqkv,
                     const float* bqkv, const void* wproj, const float* bproj, int N, int H, int W, int C,
                     void* out, void* stream);
/* with an affine (in_gamma, in_beta, in_img_stride) of the fused input norm (needs in_stats) */
int msg_la_stage_fwd_affine(int dtype, const void* x, const double* in_stats, const float* in_gamma, const float* in_beta,
                            int in_img_stride, int in_act, const void* wqkv, const float* bqkv, const void* wproj,
                            const float* bproj, int N, int H, int W, int C, void* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * layout / image helpers
 * ------------------------------------------------------------------------------------------- */
/* fp32 NCHW [N,C,H,W] -> NHWC dtype [N,H,W,Cp] (channels >= C zero-filled)  and back. */
int msg_nchw_to_nhwc(int dtype, const float* x, int N, int C, int H, int W, int Cp, void* y,
                     void* stream);
int msg_nhwc_to_nchw(int dtype, const void* x, int N, int C, int H, int W, int Cp, float* y,
                     void* stream);
/* Multi-style output blend (advanced_transform.py:206-213, direct_transform.py:155-165,
 * batch_process_images.py:306-309):  out = gain * (sum_s w[s]*ys[s] + w_x * x), optional clamp,
 * optional (v+1)/2 -> clamp(0,1) -> *255 -> uint8.  ys: S device pointers (host array) to fp32
 * tensors of `numel` elements.  out_u8 may be NULL; out_f32 may be NULL. */
int msg_blend_outputs(const float* const* ys, const float* w, int S, const float* x, float w_x,
                      float gain, int do_clip, float clip_lo, float clip_hi, long long numel,
                      float* out_f32, uint8_t* out_u8, void* stream);
/* Per-pixel multi-style blend (enhanced_local_style.py:126-176, 232-236): the weights of each output pixel come from maps.
 * ys: S (1..8) device pointers (host array) to fp32 NCHW [N,C,H,W]; x: the input image, same shape (needed when K = S+1,
 * ignored otherwise); maps: fp32 [map_batch][K][h][w] with map_batch in {1, N} (1: one map set for every image), K in {S, S+1}
 * (map S weights x), 1 <= h <= H and 1 <= w <= W.  For output pixel (n, c, i, j):
 *   1. sample m_k = bilinear(maps[n or 0][k], i, j) with F.interpolate(mode="bilinear", align_corners=False)'s source index:
 *      scale = (float)h / H, src = max(scale * (i + 0.5) - 0.5, 0), i0 = (int)src, i1 = min(i0 + 1, h - 1), t = src - i0
 *      (columns alike), interpolated as a + t * (b - a), rows first, then columns -- a constant map is returned exactly, so
 *      a 1x1 map is a per-image weight;
 *   2. normalize != 0: m_k /= sum_k m_k (all weights 0 where the sum is 0);
 *   3. v = 0; v = fmaf(m_s, ys[s], v) for s < S; v = fmaf(m_S, x, v) if K = S+1; v *= gain; optional clamp; fp32 and/or
 *      uint8 output as msg_blend_outputs.
 * With normalize = 0, constant maps equal to (w, w_x) give msg_blend_outputs' result bit for bit. */
int msg_blend_maps(const float* const* ys, int S, const float* x, const float* maps, int map_batch, int K, int h, int w,
                   int N, int C, int H, int W, int normalize, float gain, int do_clip, float clip_lo, float clip_hi,
                   float* out_f32, uint8_t* out_u8, void* stream);
/* Feathering of weight maps: scipy.ndimage.gaussian_filter(plane, sigma, mode="reflect", truncate=4.0) of each of `planes`
 * fp32 h x w planes.  Radius r = int(4 sigma + 0.5) (<= 255), taps exp(-x^2 / 2 sigma^2) normalised to sum 1 (computed in
 * double, rounded to float), vertical pass into tmp then horizontal pass into out, fp32 accumulation; indices outside [0, n)
 * reflect half-sample-symmetrically (i mod 2n, then 2n-1-i if >= n), also when r >= n.  sigma = 0 copies.
 * tmp: caller-owned [planes][h][w] fp32 workspace. */
int msg_gaussian_blur(const float* in, long long planes, int h, int w, float sigma, float* tmp, float* out, void* stream);

/* MultiScaleBlock branches at C = 64 (enhanced_generator.py:52-71: 1x1 | 3x3 dil 1 | 3x3 dil 2 | 3x3 dil 4, 64 -> 4 x 16
 * channels written as ONE 64-channel slice, bias added, optional IN statistics) as a row ring of tensor-memory accumulators:
 * every input row slab is loaded once and the three vertical taps of a dilated branch are one N = 48 MMA (csrc/msb_ring.cu).
 * x [N,H,W,Ci_total] bf16 (channels [ci_off, ci_off+64)), w_stacks bf16 [448][64] (slab.msb64_ring_weights), bias fp32 [64] or
 * NULL, y [N,H,W,Co_total] bf16 (channels [co_off, co_off+64)), stats fp64 [N][Co_total][2] with MSG_CONV_STATS. */
typedef struct {
  int dtype;                 /* MSG_BF16 */
  int N, H, W;
  int Ci_total, ci_off, Co_total, co_off;
  unsigned flags;            /* MSG_CONV_STATS */
} msg_msb_ring_desc;
int msg_msb64_ring(const msg_msb_ring_desc* d, const void* x, const void* w_stacks, const float* bias, void* y,
                   double* stats, void* stream);
/* The same for C = 64 or C = 128 input / output channels.  At C = 128 a row accumulator is 32 tensor-memory columns and the four
 * rings do not fit 512 columns: branches 1 + 2, branch 3 and branch 4 run as three launches, each with its own resident weight
 * stacks.  w_stacks: slab.msb_ring_weights(weights, C) -- per pass, per 64-channel block of the input, the stacks of the pass's
 * branches ([448][64] at C = 64, [1792][64] at C = 128); bias fp32 [C] or NULL. */
int msg_msb_ring(const msg_msb_ring_desc* d, int C, const void* x, const void* w_stacks, const float* bias, void* y,
                 double* stats, void* stream);

/* ConvTranspose2d(kernel 4, stride 2, padding 1) of the decoder (enhanced_generator.py:116-123) as a row ring of tensor-memory
 * accumulators (csrc/convt_ring.cu): one launch per horizontal output phase and 64 output channels, every input row slab loaded
 * once per launch, the four vertical taps of a horizontal tap as ONE N = 256 MMA.  Replaces the four sub-pixel phase launches of
 * msg_conv_slab for Cin in {64, 128} (the phase's weights stay resident in shared memory).
 * x [N,H,W,Ci_total] bf16 (channels [ci_off, ci_off+Cin)), w_stacks bf16 (slab.convt_ring_weights), bias fp32 [Cout] or NULL,
 * y [N,2H,2W,Co_total] bf16 (channels [co_off, co_off+Cout)), stats fp64 [N][Co_total][2] with MSG_CONV_STATS. */
typedef struct {
  int dtype;                 /* MSG_BF16 */
  int N, H, W;               /* input plane */
  int Cin, Cout;
  int Ci_total, ci_off, Co_total, co_off;
  unsigned flags;            /* MSG_CONV_STATS */
} msg_convt_ring_desc;
int msg_convt_ring(const msg_convt_ring_desc* d, const void* x, const void* w_stacks, const float* bias, void* y,
                   double* stats, void* stream);

/* Output layer of the generator fused with the InstanceNorm + ReLU + residual in front of it (enhanced_generator.py:78-84, 130-133):
 *   y = tanh(conv7x7(residual + ReLU(IN(f))) + bias), 64 -> 3 channels, fp32 NCHW out
 * as a row ring of tensor-memory accumulators (csrc/out7_ring.cu): f and residual row slabs loaded once, normalised in shared memory
 * (the apply kernel's arithmetic), the 7 vertical taps of a horizontal tap as ONE N = 112 MMA.  Inference only (a2 is not kept).
 * f [N,H,W,Cf_total] bf16 raw conv output (channels [cf_off, +64)), in_stats fp64 [N][Cs_total][2] its raw plane sums (channels
 * [cs_off, +64)), residual [N,H,W,Cr_total] bf16, w_stacks bf16 [896][64] (slab.out7_ring_weights), bias fp32 [3] or NULL,
 * y fp32 [N,3,H,W]. */
typedef struct {
  int dtype;                 /* MSG_BF16 */
  int N, H, W;
  int Cf_total, cf_off, Cr_total, cr_off, Cs_total, cs_off;
} msg_out7_ring_desc;
int msg_out7_ring(const msg_out7_ring_desc* d, const void* f, const double* in_stats, const void* residual,
                  const void* w_stacks, const float* bias, float* y, void* stream);
/* with an affine (in_gamma, in_beta, in_img_stride) of f's norm, indexed like in_stats */
int msg_out7_ring_affine(const msg_out7_ring_desc* d, const void* f, const double* in_stats, const float* in_gamma,
                         const float* in_beta, int in_img_stride, const void* residual, const void* w_stacks, const float* bias,
                         float* y, void* stream);

/* First down-sampling conv of the encoder, Conv2d(64, Cout, 4, stride 2, padding 1) (enhanced_generator.py:99-104), optionally fused
 * with the InstanceNorm + ReLU in front of it (in_stats != NULL: x is the RAW output of the previous conv and in_stats its plane sums),
 * as a row ring of tensor-memory accumulators (csrc/down_ring.cu): one launch per 64 output channels, every input row loaded once per
 * launch as its even and its odd pixels, the two vertical taps of a horizontal tap as ONE N = 128 MMA.
 * x [N,H,W,Ci_total] bf16 (channels [ci_off, +64)), H and W even; w_stacks bf16 (slab.down_ring_weights); bias fp32 [Cout] or NULL;
 * y [N,H/2,W/2,Co_total] bf16 (channels [co_off, +Cout)); stats fp64 [N][Co_total][2] with MSG_CONV_STATS. */
typedef struct {
  int dtype;                 /* MSG_BF16 */
  int N, H, W;               /* input plane */
  int Cout;
  int Ci_total, ci_off, Co_total, co_off, Cs_total, cs_off;
  unsigned flags;            /* MSG_CONV_STATS */
} msg_down_ring_desc;
int msg_down_ring(const msg_down_ring_desc* d, const void* x, const double* in_stats, const void* w_stacks, const float* bias,
                  void* y, double* stats, void* stream);
/* with an affine (in_gamma, in_beta, in_img_stride) of the fused input norm (needs in_stats), indexed like in_stats */
int msg_down_ring_affine(const msg_down_ring_desc* d, const void* x, const double* in_stats, const float* in_gamma,
                         const float* in_beta, int in_img_stride, const void* w_stacks, const float* bias, void* y,
                         double* stats, void* stream);

/* uint8 pre-processing on the device (batch_process_images.py:193-205, 287-291): paste the [N,h,w,3] uint8 images (PIL layout) at
 * (off_y, off_x) on an HxW canvas filled with `fill` (the reference's white canvas), then ToTensor + Normalize(0.5, 0.5):
 * out fp32 NCHW [N,3,H,W] = (v / 255 - 0.5) / 0.5.  canvas (optional, may be NULL): the pasted uint8 canvas [N,H,W,3].
 * With h == H, w == W and zero offsets it is the plain uint8 -> normalised conversion. */
int msg_u8_canvas_to_nchw(const uint8_t* img, int N, int h, int w, int H, int W, int off_y, int off_x, int fill,
                          float* out, uint8_t* canvas, void* stream);
/* "simple" mode strength blend in uint8 space (batch_process_images.py:304-310, gan_login_gui.py:826):
 * out = uint8(clip(orig * (1 - s) + styled * s, 0, 255)), float64 arithmetic, truncating conversion.
 * orig / out: NHWC uint8 [N,H,W,3]; styled: NCHW uint8 [N,3,H,W] (msg_blend_outputs' uint8 result). */
int msg_u8_strength_blend(const uint8_t* orig_nhwc, const uint8_t* styled_nchw, int N, int H, int W, double strength,
                          uint8_t* out_nhwc, void* stream);

/* ---------------------------------------------------------------------------------------------
 * losses (enhanced_train.py:49-52): mean-reduced MSE / L1, forward value and input gradient.
 * loss_out: device fp32 scalar, ACCUMULATED into (+= scale * mean(...)); grad_a = scale*d/da.
 * b may be NULL with b_const used instead (ones_like / zeros_like targets, :72-79,100-101).
 * ------------------------------------------------------------------------------------------- */
int msg_mse_loss(const float* a, const float* b, float b_const, long long n, float scale,
                 float* loss_out, float* grad_a, void* stream);
int msg_l1_loss(const float* a, const float* b, float b_const, long long n, float scale,
                float* loss_out, float* grad_a, float* grad_b, void* stream);

/* fused Adam (enhanced_train.py:36-43): one launch over a flat fp32 parameter buffer.
 * grad_scale multiplies the gradient first (1/world_size after the NCCL sum-allreduce). */
int msg_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                  float beta2, float eps, int step, float grad_scale, void* stream);

/* as msg_adam_step with the step count kept in device memory: *step_dev is incremented, then used for the bias corrections
 * (host double-precision pow of msg_adam_step restated on the device).  For CUDA-graph replays of a whole train step. */
int msg_adam_step_dev(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                      float beta2, float eps, int* step_dev, float grad_scale, void* stream);

/* spectral norm (old-style torch.nn.utils.spectral_norm, enhanced_generator.py:269-271):
 * one power iteration on W[rows][cols] (fp32), updating u[rows], v[cols] in place, then
 * sigma = u^T W v written to *sigma.  do_power_iter=0 (eval) only computes sigma. */
int msg_spectral_norm(const float* w, int rows, int cols, float* u, float* v, int do_power_iter,
                      float eps, float* sigma, void* stream);
/* gradient through weight = weight_orig / sigma:
 * dw_orig += (dw - <dw, w_orig>/sigma * u v^T) / sigma  */
/* the same for up to MSG_SN_MAX_BATCH weights in one launch (all seven convs of one discriminator forward,
 * enhanced_generator.py:269-271): problem i = (w[i], rows[i], cols[i], u[i], v[i]) -> *sigma[i]. */
#define MSG_SN_MAX_BATCH 8
typedef struct {
  const float* w[MSG_SN_MAX_BATCH];
  float* u[MSG_SN_MAX_BATCH];
  float* v[MSG_SN_MAX_BATCH];
  float* sigma[MSG_SN_MAX_BATCH];
  int rows[MSG_SN_MAX_BATCH];
  int cols[MSG_SN_MAX_BATCH];
  int n;
} msg_sn_batch;
int msg_spectral_norm_batched(const msg_sn_batch* b, int do_power_iter, float eps, void* stream);

int msg_spectral_norm_bwd(const float* dw, const float* w_orig, const float* u, const float* v,
                          const float* sigma, int rows, int cols, float* dw_orig, float* scratch,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gram matrix + style loss (north_star addition; not in the reference, SURVEY.md F5).
 * feat: [N,H,W,C] dtype.  gram: fp32 [N][C][C] = F F^T / (C*H*W).
 * msg_gram_loss_fwd: loss += scale * mean((G - target)^2); keeps G for the backward.
 * msg_gram_loss_bwd: dfeat = scale * 2/(N*C*C) * 2/(C*H*W) * (G - target) . F   (written, dtype).
 * ------------------------------------------------------------------------------------------- */
int msg_gram(int dtype, const void* feat, int N, long long HW, int C, float* gram, void* stream);
int msg_gram_loss_fwd(int dtype, const void* feat, int N, long long HW, int C, const float* target,
                      float scale, float* gram, float* loss_out, void* stream);
int msg_gram_loss_bwd(int dtype, const void* feat, int N, long long HW, int C, const float* gram,
                      const float* target, float scale, void* wscratch /* dtype [N][C][C] */,
                      void* dfeat, void* stream);
/* 2x2 max pool (VGG trunk) fwd/bwd on NHWC. */
int msg_maxpool2x2_fwd(int dtype, const void* x, int N, int H, int W, int C, void* y, void* stream);
int msg_maxpool2x2_bwd(int dtype, const void* x, const void* dy, int N, int H, int W, int C,
                       void* dx, void* stream);
/* elementwise backward of an activation applied in a conv epilogue: dx = dy * act'(y). */
int msg_act_bwd(int dtype, const void* y, const void* dy, long long n, int act, void* dx,
                void* stream);
/* tanh backward on the fp32 NCHW image: dz (NHWC dtype, Cp channels) = dy * (1 - y^2). */
int msg_tanh_bwd_nchw(int dtype, const float* y, const float* dy, int N, int C, int H, int W,
                      int Cp, void* dz, void* stream);
/* out = a + b (dtype tensors, n elements); used to sum gradient branches. */
int msg_add(int dtype, const void* a, const void* b, long long n, void* out, void* stream);
/* mean over the H*W plane of a [N,HW,C] tensor -> fp32 [N][C]  (AdaptiveAvgPool2d(1),
 * enhanced_generator.py:257) and its backward (broadcast of dy/HW). */
int msg_avgpool_fwd(int dtype, const void* x, int N, long long HW, int C, float* y, void* stream);
int msg_avgpool_bwd(int dtype, const float* dy, int N, long long HW, int C, void* dx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSG_B200_H_ */
