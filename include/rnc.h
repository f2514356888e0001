/* rnc.h — C ABI of librnc.so: the B200 (sm_100a) kernels behind RAFT-NCUP's per-iteration hot path.
 *
 * The reference (abdo-eldesokey/RAFT-NCUP @ 51ac387) has NO native layer: every op below is a chain of
 * PyTorch eager calls.  Each entry point therefore cites the reference *Python* interface it replaces
 * (file:line under /root/reference).  INTEGRATION.md shows the ctypes stub a maintainer of the reference
 * would add at each call site.
 *
 * Conventions
 *   - every function returns 0 (RNC_OK) or a negative rnc_status; nothing throws across the boundary
 *   - all pointers are DEVICE pointers to caller-owned buffers (e.g. torch tensor.data_ptr()); no hidden
 *     allocation, no global mutable state, re-entrant; work is enqueued on `stream` (a cudaStream_t passed
 *     as void*) and the call returns immediately
 *   - "NCHW" tensors are the reference's own layout; "CL" = channel-last [B][H][W][C] fp32, the resident
 *     layout of the 1/8-resolution activations inside the iteration loop
 */
#ifndef RNC_H_
#define RNC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  RNC_OK = 0,
  RNC_ERR_BAD_SHAPE = -1,     /* dimension <= 0, unsupported radius/levels/channel count */
  RNC_ERR_BAD_POINTER = -2,   /* null or misaligned (16 B) pointer */
  RNC_ERR_UNSUPPORTED = -3,   /* valid request this build does not implement */
  RNC_ERR_CUDA = -4,          /* launch failed; see rnc_last_cuda_error() */
  RNC_ERR_WORKSPACE = -5      /* workspace too small */
} rnc_status;

/* Library identity / diagnostics. */
int rnc_abi_version(void);                 /* bumps on any signature change (now 11) */
const char* rnc_build_info(void);          /* e.g. "sm_100a nvcc 12.9" */
const char* rnc_status_string(int status);
int rnc_last_cuda_error(void);             /* cudaError_t of the last failed launch on this thread */
/* Number of kernels launched by this library on the calling thread since the last reset (bench.py's
 * `gpu_launches` claim is read from here). */
long long rnc_launch_count(void);
void rnc_launch_count_reset(void);

/* ------------------------------------------------------------------------------------------------
 * A1  CorrBlock.__init__  (core/corr.py:7-21, 47-55)
 * Replaces the all-pairs matmul + avg_pool2d pyramid.  Nothing quadratic is built: fmap1 is transposed to
 * CL and fmap2 is transposed + average-pooled (floor mode, 2x2) into a `levels`-deep CL pyramid; pooling
 * commutes with the dot product so lookups against it equal lookups into the reference's 4-D pyramid.
 *   fmap1, fmap2 : [B][D][H][W] fp32 NCHW
 *   f1_cl        : [B][H*W][D]
 *   f2_pyr       : level l at element offset rnc_pyramid_offset(B,D,H,W,l), shape [B][H>>l][W>>l][D]
 */
size_t rnc_pyramid_offset(int B, int D, int H, int W, int level);   /* in elements; level==levels -> total */
int rnc_fmap_prepare(const float* fmap1, const float* fmap2, int B, int D, int H, int W, int levels,
                     float* f1_cl, float* f2_pyr, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A2/A3  CorrBlock.__call__ + bilinear_sampler  (core/corr.py:23-44, core/utils/utils.py:59-73)
 * Fused multi-scale lookup straight from the feature maps.
 *   coords : [B][2][H][W] fp32 NCHW (channel 0 = x, 1 = y), level-0 pixel units
 *   out    : layout 0 -> [B][L*(2r+1)^2][H][W]   (the reference's return value, corr.py:44)
 *            layout 1 -> CL [B][H][W][ldo], channels [0, L*(2r+1)^2) written, ldo >= that
 *   channel k = l*(2r+1)^2 + i*(2r+1) + j  samples level l at (cx/2^l + i - r, cy/2^l + j - r): the slow
 *   window index offsets x (corr.py:31-37).  Bilinear, zero outside, scaled by 1/sqrt(D).
 * Supported: D % 32 == 0, radius == 4 (the only value the reference's models use, raft_nc_dbl.py:41), 1 <= levels <= 4.
 */
int rnc_corr_lookup_fwd(const float* f1_cl, const float* f2_pyr, const float* coords,
                        int B, int D, int H, int W, int levels, int radius,
                        float* out, int layout, int ldo, void* stream);

/* Same lookup, written as exact fp16 hi/lo split planes (CL [B][H][W][ldo] halves each; value = hi + lo): the operand
 * format of rnc_conv2d_umma_fwd, so the 1x1 convc1 (update.py:82,90) consumes it without a conversion pass. */
int rnc_corr_lookup_split_fwd(const float* f1_cl, const float* f2_pyr, const float* coords,
                              int B, int D, int H, int W, int levels, int radius,
                              void* out_hi, void* out_lo, int ldo, int lvl_stride, void* stream);
/* lvl_stride: channels reserved per pyramid level in the output row (>= 81; level l starts at l*lvl_stride, the
 * channels [81, lvl_stride) of each level are written as zeros).  The tensor-core path uses 88 so that every 8-channel
 * group is one aligned 16-byte store and convc1's K stays 6 blocks of 64.
 * Channel order of the split planes inside a level ("resident order"; only convc1 consumes them, with its weight rows
 * permuted to match): tap (i, j) -> j*8 + i for i < 8, tap (8, j) -> 72 + j  — a pixel's 8 values of one window row are
 * one aligned 16-byte group.  The reference order k = i*9 + j is what rnc_corr_lookup_fwd returns. */

/* Tensor-core version of the lookup (tcgen05 + TMA; same reference code, corr.py:7-55 + utils.py:59-73).
 *   f1h_cl / f2h_pyr : the CL feature map / pyramid of rnc_fmap_prepare rounded once to halves (rnc_f32_to_f16), same
 *                      element offsets (rnc_pyramid_offset)
 *   f1_cl / f2_pyr   : the fp32 originals, used by the exact CUDA-core kernel for tiles whose lookup windows do not
 *                      fit the fixed per-level boxes (incoherent flow) — results never depend on a coherence assumption
 *   out_hi / out_lo  : CL split halves planes [B][H][W][ldo] (value = hi + lo)
 *   workspace        : rnc_corr_lookup_umma_workspace_bytes(B,H,W) bytes of device memory (per-tile fallback flags)
 * Supported: D == 256, levels == 4, radius == 4.
 */
size_t rnc_corr_lookup_umma_workspace_bytes(int B, int H, int W);
int rnc_corr_lookup_umma_fwd(const void* f1h_cl, const void* f2h_pyr, const float* f1_cl, const float* f2_pyr,
                             const float* coords, int B, int D, int H, int W, int levels, int radius,
                             void* out_hi, void* out_lo, int ldo, int lvl_stride, void* workspace, size_t workspace_bytes,
                             void* stream);   /* lvl_stride must be 88; resident channel order (above); out_hi/out_lo
                                                 16-byte aligned, ldo % 8 == 0: the tiles leave through TMA stores */
/* fp32 -> fp16 (round to nearest), n % 4 == 0. */
int rnc_f32_to_f16(const float* src, void* dst, size_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A5..A8  update block convolutions  (core/update.py:6-14, 33-60, 79-97, 114-141)
 * One generic channel-last convolution with the update block's fusions expressed as epilogues.
 * The input is the virtual concatenation of up to two CL segments (replaces torch.cat, update.py:46,49,95,132).
 * weight is pre-packed [KH*KW][Cin][CoutPad] fp32 (CoutPad = Cout rounded up to 64), bias [CoutPad].
 */
typedef enum {
  RNC_EPI_LINEAR = 0,   /* out = acc + bias                                                     */
  RNC_EPI_RELU = 1,     /* out = relu(acc + bias)                       update.py:90-96, 14     */
  RNC_EPI_SIGMOID = 2,  /* out = sigmoid(acc + bias)                                            */
  RNC_EPI_GRU_ZR = 3,   /* Cout = 2*C: ch<C: aux0[p][ch] = z = sigmoid(.)                       */
                        /*             ch>=C: out[p][ch-C] = sigmoid(.) * h[p][ch-C]   update.py:47-49 */
  RNC_EPI_GRU_Q = 4,    /* q = tanh(.); h[p][ch] = (1-z)*h + z*q with z = aux0       update.py:49-50 */
  RNC_EPI_RELU_FLOW = 5,/* RELU, and channels [Cout, Cout+2) of out receive flow = coords1-coords0 (update.py:97);
                           aux0 = coords1 NCHW [B][2][H][W]                                     */
  RNC_EPI_RELU_ADD_RELU = 6, /* relu(res + relu(acc + bias)): residual block tail, extractor.py:48-55 (umma only) */
  RNC_EPI_TANH_RELU = 7,     /* ch < Cout/2: tanh (-> out_f32 and split), else relu (-> split): raft_nc_dbl.py:138-140 (umma only) */
  RNC_EPI_FLOW_DELTA = 8     /* Cout = 2 (FlowHead.conv2, update.py:10,14): aux0 = coords1 NCHW [B][2][H][W] += (acc + bias)
                                (raft_nc_dbl.py:157); out_f32, if given, receives delta_flow NCHW (umma only) */
} rnc_epilogue;

/* rnc_conv_umma_desc.flags */
#define RNC_CONV_NO_HALO 1          /* force one A tile per filter tap (disable the row/column halo sharing) */
#define RNC_CONV_BASE_OFFSET 2      /* reserved (round-1 debug switch for the descriptor base_offset; ignored)  */
#define RNC_CONV_AUX_BLOCKED 16     /* aux0 (z gate) and add are tile-blocked: element (tile, channel c, row r) at ((tile*ld + c)*128 + r) */
#define RNC_CONV_OUT_BLOCKED 32     /* RNC_EPI_LINEAR: out_f32 in the same tile-blocked layout (produces an `add` operand)          */
#define RNC_CONV_NO_PAIR 8          /* never use the CTA-pair (cta_group::2) form for this call */
#define RNC_CONV_SPLIT_N 4          /* 256-column layers as two 128-column items per pixel tile (double-buffered TMEM) */
#define RNC_CONV_WINDOW 128        /* in0 is a sliding-window view of a padded plane, see rnc_conv_umma_desc.win_pitch */
#define RNC_CONV_TF32 64            /* operands are fp32 hi/lo planes consumed as TF32 (tcgen05 kind::tf32, K = 8): value = hi + lo with
                                     * hi = tf32(value), 3 MMAs per K step as in the fp16 form but with fp32's exponent range — the
                                     * training path's layers (output gradients underflow the fp16 split).  The in / w pointers address float
                                     * planes, ld / ktot count floats, K blocks hold 32 channels, only out_f32 is written. */

typedef struct {
  const float* in0; int c0; int ld0;   /* segment 0: channels [0,c0), pixel stride ld0 floats   */
  const float* in1; int c1; int ld1;   /* segment 1 (optional, c1 = 0 if absent)                */
  const float* weight; const float* bias;
  float* out; int ldo;                 /* CL output, pixel stride ldo                           */
  float* h; int ldh;                   /* GRU hidden state (read; written by GRU_Q)             */
  float* aux0; int ldaux;              /* z buffer (GRU) or coords1 (RELU_FLOW)                 */
  int B, H, W;
  int cout;                            /* logical Cout (<= CoutPad)                             */
  int kh, kw;                          /* odd; zero padding kh/2, kw/2 (all reference convs)    */
  int epilogue;                        /* rnc_epilogue                                          */
} rnc_conv_desc;

int rnc_conv2d_cl_fwd(const rnc_conv_desc* desc, void* stream);

/* Tensor-core version of rnc_conv2d_cl_fwd (same reference code, same epilogues): tcgen05.mma on fp16 hi/lo split
 * operands with fp32 accumulation in TMEM (3 MMAs per K step: hi*hi + hi*lo + lo*hi), TMA-staged tiles.
 * Activations live as two CL planes of halves (value = hi + lo); weights are pre-split and pre-scaled by a power of two:
 *   w_hi/w_lo : [coutpad][ktot] halves, ktot = kh*kw * nblocks * 64, K index = (tap * nblocks + block) * 64 + c,
 *               blocks enumerate 64-channel slices of segment 0 then segment 1, zero rows for channels beyond Cin
 *   unscale   : 1 / (weight scale); out = act(acc * unscale + bias)
 * Outputs: out_f32 (CL fp32) and/or out_hi/out_lo (CL split halves); either may be NULL.
 *   GRU_ZR : z -> aux0 (fp32), r*h -> out_hi/out_lo;   GRU_Q : h (fp32, in place) and its split copy -> out_hi/out_lo
 *   RELU_FLOW: split output, flow appended at channels [cout, cout+2); aux0 = coords1 NCHW
 */
typedef struct {
  const void* in0_hi; const void* in0_lo; int c0; int ld0;
  const void* in1_hi; const void* in1_lo; int c1; int ld1;
  const void* w_hi; const void* w_lo; int ktot; int coutpad;
  const float* bias; float unscale;
  float* out_f32; int ldo_f32;
  void* out_hi; void* out_lo; int ldo_split;
  float* h; int ldh;
  float* aux0; int ldaux;
  int B, H, W;
  int cout;
  int kh, kw;
  int epilogue;
  int stride;                          /* 1 (or 0) | 2: output pixel (y,x) reads input (stride*y + ky - kh/2, ...) */
  int hin, win;                        /* input height/width (0 -> same as H, W)                                    */
  const float* res; int ldres;         /* residual (fp32 CL at output resolution) for RELU_ADD_RELU                 */
  int flags;                           /* RNC_CONV_*                                                                 */
  double* stats;                       /* optional (RNC_EPI_LINEAR + out_f32 only): [B][cout][2] sum / sum of squares of the
                                        * outputs, ACCUMULATED (caller keeps it zeroed: rnc_instnorm_finalize re-zeroes) */
  const float* add; int ldadd;         /* optional: fp32 [B*H*W][ldadd] added to the pre-activation (after bias), e.g. the
                                        * hoisted contribution of input channels that do not change between calls */
  int win_pitch;                       /* RNC_CONV_WINDOW (kw = 1, stride 2, c1 = 0): position x of input row y exposes the c0
                                        * consecutive halves that start at element y*win_pitch + x*ld0 of in0 (ld0 < c0: the
                                        * windows overlap; the TMA unit builds the im2col rows); win = positions per row (one
                                        * per output column), hin = rows, the stride applies to rows only. Used by the encoders'
                                        * 7x7/2 stem: a [hin][win_pitch/4][4] zero-padded pixel plane, 16-pixel windows, ld0 = 8 */
} rnc_conv_umma_desc;

/* Pixel tiles (128 output pixels each) a layer of this shape is cut into: a tile-blocked tensor with ld channels has
 * rnc_conv_umma_tiles(...) * ld * 128 floats; the tiling depends on (kh, kw, stride, H, W, flags & RNC_CONV_NO_HALO) only.
 * Tile shape TW x TH px (stride 1, no RNC_CONV_NO_HALO): 128 x 1 if kw > 1 and W > 64; 16 x 8 if kw == 1 < kh, W >= 16 and
 * H >= 8; otherwise (and for stride 2 or RNC_CONV_NO_HALO) TW = the smallest power of two >= W in [8, 128], TH = 128 / TW.
 * Tile t = (b * ceil(H/TH) + ty) * ceil(W/TW) + tx holds pixel (y, x) = (ty*TH + r / TW, tx*TW + r % TW) at row r. */
long long rnc_conv_umma_tiles(int kh, int kw, int stride, int B, int H, int W, int flags);
int rnc_conv2d_umma_fwd(const rnc_conv_umma_desc* desc, void* stream);

/* fp32 CL [M][lds] channels [0,C) -> split halves planes [M][ldd] at channel offset ch_off (hi + lo == value exactly
 * when |value| <= 65504). */
int rnc_f32_to_split(const float* src, int lds, int C, long long M, void* dst_hi, void* dst_lo, int ldd, int ch_off,
                     void* stream);

/* fp32 CL [M][lds] channels [0,C) -> TF32 hi/lo planes of floats [M][ldd] at channel offset ch_off: hi = value rounded to TF32
 * (cvt.rna), lo = value - hi (operands of RNC_CONV_TF32 layers; hi + lo reproduces the value to ~2^-21). */
int rnc_f32_to_tf32_split(const float* src, int lds, int C, long long M, float* dst_hi, float* dst_lo, int ldd, int ch_off,
                          void* stream);

/* convf1: Conv2d(2,128,7,padding=3)+ReLU on flow = coords1 - coords0 (update.py:83,92).
 * coords1 NCHW [B][2][H][W]; weight packed [49][2][Cout]; out CL. */
int rnc_conv_flow7x7_fwd(const float* coords1, const float* weight, const float* bias, int B, int H, int W,
                         int cout, float* out, int ldo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * C6  BasicEncoder pieces (core/extractor.py:118-192) that are not wide convolutions; the 3x3/1x1 layers run on
 * rnc_conv2d_umma_fwd (stride 1/2, RELU / RELU_ADD_RELU / TANH_RELU epilogues).
 */
/* Image normalisation 2*(x/255)-1 (raft_nc_dbl.py:118-119) + conv1 = Conv2d(3,64,7,stride=2,padding=3) (extractor.py:135,171).
 * img NCHW [N][3][Hin][Win] raw 0..255; weight [147 = (c*7+ky)*7+kx][64]; bias [64]; out CL [N][ceil(Hin/2)][ceil(Win/2)][64]
 * as fp32 and/or split halves; relu != 0 applies ReLU (norm folded into the weights). */
int rnc_stem_conv7x7s2_fwd(const float* img, const float* weight, const float* bias, int N, int Hin, int Win, int relu,
                           float* out_f32, void* out_hi, void* out_lo, void* stream);
/* The same layer on the tensor cores: this call normalises the image and repacks it as a zero-padded pixel plane of split
 * halves [N][Hin][pitch_px][4] (pixel p = image column p - 3, channel 3 = 0; pitch_px even, >= Win + 6; the caller keeps
 * >= 16 zero pixels after the last row); rnc_conv2d_umma_fwd then reads it as a sliding-window view (RNC_CONV_WINDOW:
 * c0 = 64 = 16 pixels x 4, ld0 = 8, win_pitch = 4*pitch_px, kh = 7, kw = 1, stride 2) with the 7x7x3 filter laid out as
 * [64][7 rows][16 px x 4 ch] (zeros for px >= 7 and channel 3): the TMA unit builds the im2col rows, no copy. */
int rnc_stem_window_prep(const float* img, int N, int Hin, int Win, int pitch_px, void* out_hi, void* out_lo, void* stream);
/* nn.InstanceNorm2d (no affine, biased variance; extractor.py:28-33,128-129) statistics of x CL fp32 [N][P][C], C <= 128:
 * stats = fp64 scratch [N][C][2]; mean_rstd = [N][C][2] floats (mean, 1/sqrt(var+eps)). */
int rnc_instnorm_stats(const float* x, int N, int P, int C, float eps, double* stats, float* mean_rstd, void* stream);
/* Second half of rnc_instnorm_stats when the sums were accumulated elsewhere (rnc_conv_umma_desc.stats): stats [N][C][2]
 * fp64 sums over P positions -> mean_rstd, then stats is zeroed for the next producer. */
int rnc_instnorm_finalize(double* stats, int N, int P, int C, float eps, float* mean_rstd, void* stream);
/* apply: mode 0: norm(x) -> out_f32;  1: relu(norm(x));  2: relu(res + relu(norm(x)))  (ResidualBlock.forward,
 * extractor.py:48-56); outputs fp32 and/or split halves, all CL [N][P][C]. */
int rnc_instnorm_apply(const float* x, const float* mean_rstd, const float* res, int N, int P, int C, int mode,
                       float* out_f32, void* out_hi, void* out_lo, void* stream);
/* relu(a + b) on n fp32 elements -> fp32 (optional) + split halves (block tail when the downsample branch has its own norm). */
int rnc_add_relu_split(const float* a, const float* b, size_t n, float* out_f32, void* out_hi, void* out_lo, void* stream);
/* Pooling half of rnc_fmap_prepare for feature maps that are already CL: fills levels 1..levels-1 of f2_pyr from level 0. */
int rnc_fmap_pyramid(float* f2_pyr, int B, int D, int H, int W, int levels, void* stream);

/* convf1 with split-halves CL output (feeds the tensor-core convf2). */
int rnc_conv_flow7x7_split_fwd(const float* coords1, const float* weight, const float* bias, int B, int H, int W,
                               int cout, void* out_hi, void* out_lo, int ldo, void* stream);

/* FlowHead.conv2 (update.py:10,14) fused with `coords1 = coords1 + delta_flow` (raft_nc_dbl.py:157):
 * in CL [B][H][W][cin]; weight packed [9][cin][2]; delta (optional, may be NULL) and coords1 NCHW [B][2][H][W]. */
int rnc_flow_head2_fwd(const float* in, int cin, int ldi, const float* weight, const float* bias,
                       int B, int H, int W, float* delta, float* coords1, void* stream);

/* convf1 = Conv2d(2,128,7,padding=3) on flow = coords1 - grid (update.py:83,93-94), first half of the tensor-core
 * formulation: writes, for every pixel, its zero-padded 7x7x2 flow neighbourhood as 98 (+30 zero) split halves,
 * column k = 2*(7*ky+kx)+c, rows of ld >= 128 halves; a 1x1 rnc_conv2d_umma_fwd with the [128][98] weight finishes it. */
int rnc_flow_im2col7_split_fwd(const float* coords1, int B, int H, int W, void* out_hi, void* out_lo, int ld, void* stream);

/* FlowHead.conv2 (update.py:10,14), second half of the tensor-core formulation: `taps` [B*H*W][ldt] fp32 holds, for every
 * pixel q, the 18 values W[o][:, ky, kx] . in[q] at column 2*(3*ky+kx)+o (a 1x1 convolution by rnc_conv2d_umma_fwd, K =
 * cin instead of 9*cin); this sums the in-image 3x3 neighbours (zero padding), adds bias[2] (device), writes delta
 * (optional, NCHW [B][2][H][W]) and does `coords1 = coords1 + delta_flow` (raft_nc_dbl.py:157). */
int rnc_flow_tap_gather_fwd(const float* taps, int ldt, const float* bias, int B, int H, int W, float* delta, float* coords1,
                            void* stream);

/* coords_grid / initialize_flow (core/utils/utils.py:76-79, raft_nc_dbl.py:83-90) (+ optional flow_init, :144-145).
 * coords1 = grid (+ flow_init);  flow_init may be NULL. */
int rnc_coords_init(float* coords1, const float* flow_init, int B, int H, int W, void* stream);
/* flow = coords1 - grid  -> NCHW [B][2][H][W]  (raft_nc_dbl.py:152,170). */
int rnc_coords_to_flow(const float* coords1, float* flow, int B, int H, int W, void* stream);

/* Warm start: forward_interpolate (core/utils/utils.py:28-56; evaluate.py:38-40): push every pixel along its flow,
 * keep samples landing strictly inside the image, give each grid point the flow of its nearest kept sample
 * (scipy griddata 'nearest', fill 0).  flow, out: NCHW [B][2][H][W]. */
int rnc_forward_interpolate_fwd(const float* flow, int B, int H, int W, float* out, void* stream);

/* Layout plumbing between the reference's NCHW tensors and the resident CL buffers. */
int rnc_nchw_to_cl(const float* src, int B, int C, int H, int W, float* dst, int ldd, int ch_off, void* stream);
int rnc_cl_to_nchw(const float* src, int lds, int ch_off, int B, int C, int H, int W, float* dst, void* stream);

/* ------------------------------------------------------------------------------------------------
 * U1  RAFT.upsample_flow, convex combination  (core/raft.py:73-84)
 *   flow NCHW [B][2][H8][W8]; mask CL [B][H8][W8][ldm] with 576 logits (c = k*64 + sy*8 + sx, k = ky*3+kx),
 *   already scaled by 0.25 (update.py:140); out NCHW [B][2][8*H8][8*W8].
 */
int rnc_convex_upsample_fwd(const float* flow, const float* mask, int ldm, int B, int H8, int W8,
                            float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * U2  RAFT.upsample_flow prologue (raft_nc_dbl.py:110): x4 = nearest-x2 of flow_lr = coords1 - grid.
 *   coords1 NCHW [B][2][H8][W8] -> x4 NCHW [B][2][2*H8][2*W8]
 */
int rnc_flow_x2_fwd(const float* coords1, int B, int H8, int W8, float* x4, void* stream);

/* U3 (input staging)  upsampler.py:150,155 — builds the weights-net input at 1/4 resolution, CL [B][2*H8][2*W8][ldo]:
 *   channels 0,1 = x_lowres (NCHW [B][2][2*H8][2*W8]); channels 2..2+C = guidance (net, CL [B][H8][W8][ldg]) resized
 *   'area' H8 -> 2*H8, which for an integer x2 upscale is replication; channels >= 2+C are zero-filled.
 */
int rnc_ncup_guidance_fwd(const float* x_lowres, const float* net, int ldg, int C, int B, int H8, int W8,
                          float* out, int ldo, void* stream);

/* The same staging written directly as split halves planes [B][2*H8][2*W8][ldo] (ldo % 8 == 0, channels >= 2+C zero): the
 * operand of the tensor-core weights net, without the fp32 intermediate. */
int rnc_ncup_guidance_split_fwd(const float* x_lowres, const float* net, int ldg, int C, int B, int H8, int W8,
                                void* out_hi, void* out_lo, int ldo, void* stream);

/* U4 tail: Simple.out (1x1 conv 32->2) + sigmoid (interp_weights_est.py:37,47; upsampler.py:44-46):
 *   in CL [B][H4][W4][cin] -> conf NCHW [B][2][H4][W4]. weight packed [cin][2]. */
int rnc_conf_head_fwd(const float* in, int cin, int ldi, const float* weight, const float* bias,
                      int B, int H4, int W4, float* conf, void* stream);

/* ------------------------------------------------------------------------------------------------
 * U3/U5/U6  NConvUpsampler.forward + NConvUNet.forward (live path) + NConv2d.forward
 *           (core/upsampler.py:143-177,179-210; core/nconv_modules.py:106-136,164-199)
 * Fused zero-stuff (scale 4, offset 2) + 4 normalized convolutions + the x8 of raft_nc_dbl.py:161.
 *   x_lowres: NCHW [B][2][H4][W4]   low-resolution data (in RAFT: nearest-x2 flow at 1/4 resolution)
 *   conf    : NCHW [B][2][H4][W4]   sigmoid output of the weights net
 *   wts_host: HOST pointer to 224 floats = softplus_{beta=10}(weight_p) of nconv_in[2,1,5,5], nconv_x2.0[2,2,5,5],
 *             decoder.0[2,4,3,3], nconv_out[1,2,1,1] in that order (nconv_modules.py:250-264).  They are copied
 *             into the kernel's parameter bank at launch (read before the call returns), so the call stays
 *             re-entrant with no device-side global state.
 *   out     : NCHW [B][2][4*H4][4*W4] = out_scale * NConvUNet output  (out_scale = 8 in RAFT, raft_nc_dbl.py:161)
 */
int rnc_ncup_fwd(const float* x_lowres, const float* conf, const float* wts_host, int B, int H4, int W4,
                 float out_scale, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A3  bilinear_sampler  (core/utils/utils.py:59-73) as a standalone operator: grid_sample(align_corners=True, bilinear,
 * zero padding) with the grid in pixel coordinates.  img NCHW [N][C][H][W]; coords [N][h][w][2] = (x, y); out NCHW
 * [N][C][h][w]; mask (optional, may be NULL) [N][h][w][1] as utils.py:69-71.  H, W >= 2 (the reference divides by W-1).
 */
int rnc_bilinear_sample_fwd(const float* img, const float* coords, int N, int C, int H, int W, int h, int w,
                            float* out, float* mask, void* stream);

/* ------------------------------------------------------------------------------------------------
 * U6  NConv2d.forward  (core/nconv_modules.py:164-199) — ONE normalized-convolution layer, the operator seam
 *     `NConv2d((data, conf)) -> (y, conf_out)`, and the per-layer form the training path differentiates through
 *     (the inference path runs the fused chain rnc_ncup_fwd instead).
 *   data, conf : NCHW [N][Cin][H][W] fp32;  weight: [Cout][Cin][kh][kw] fp32 = softplus_{beta=10}(weight_p)
 *                (nconv_modules.py:250-264; the caller applies it), zero padding k/2, stride 1, no bias
 *   y = conv(data*conf, W) / (conv(conf, W) + eps),   conf_out = conv(conf, W) / sum_{i,ky,kx} W[o]
 * Supported: Cin, Cout <= 4, odd kh, kw <= 7.
 */
int rnc_nconv2d_fwd(const float* data, const float* conf, const float* weight, int N, int Cin, int Cout, int H, int W,
                    int kh, int kw, float eps, float* y, float* conf_out, void* stream);
/* Backward of rnc_nconv2d_fwd (autograd of nconv_modules.py:169-194: quotient rule through num/(den+eps), confidence
 * propagation incl. its dependence on sum(W)).  g_y / g_conf_out: upstream gradients (either may be NULL = zero);
 * g_data, g_conf, g_weight ([Cout][Cin][kh][kw], w.r.t. the POSITIVE kernel; the caller chains softplus'): outputs, each
 * may be NULL.  workspace: rnc_nconv2d_bwd_workspace_bytes(N,Cout,H,W) bytes, ZERO-INITIALISED by the caller before its
 * first use (the call leaves its accumulators zeroed again). */
size_t rnc_nconv2d_bwd_workspace_bytes(int N, int Cout, int H, int W);
int rnc_nconv2d_bwd(const float* data, const float* conf, const float* weight, const float* y, const float* conf_out,
                    const float* g_y, const float* g_conf_out, int N, int Cin, int Cout, int H, int W, int kh, int kw,
                    float eps, float* g_data, float* g_conf, float* g_weight, void* workspace, size_t workspace_bytes,
                    void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training path (train.py:203-227; SURVEY.md §8f-3, Appendix G): backward kernels, exact fp32, and the TF32x3 tensor-core
 * form of the convolution weight gradient.
 *
 * Gradient of CorrBlock.__call__ (core/corr.py:23-44; the reference back-propagates through the stored 4-D pyramid) w.r.t.
 * the feature maps.  coords are detached (raft_nc_dbl.py:149): no gradient flows to them.
 *   g_out    : CL [B][H][W][ldg], channels [0, 324) in the reference order k = l*81 + i*9 + j
 *   g_f1     : CL [B][H*W][D], written
 *   g_f2_pyr : pyramid layout of rnc_fmap_prepare, ACCUMULATED with atomics — the caller zero-fills it; finish with
 *              rnc_pyramid_pool_bwd, which folds levels 3..1 into level 0 (adjoint of the 2x2 average pooling,
 *              core/corr.py:18-21 applied to features) so that level 0 holds d loss / d fmap2 (CL)
 */
int rnc_corr_lookup_bwd(const float* f1_cl, const float* f2_pyr, const float* coords, const float* g_out, int ldg,
                        int B, int D, int H, int W, int levels, int radius, float* g_f1, float* g_f2_pyr, void* stream);
int rnc_pyramid_pool_bwd(float* g_f2_pyr, int B, int D, int H, int W, int levels, void* stream);

/* Weight and bias gradient of a channel-last convolution y = conv(x, w) + b (stride 1 or 2, zero padding k/2):
 *   x  : CL [B][Hin][Win][ldx], cin % 4 == 0;   gy : CL [B][ceil(Hin/s)][ceil(Win/s)][ldg] = d loss / d y
 *   gw : [kh*kw][cin][ldw] fp32 (the packing of rnc_conv2d_cl_fwd's weight), ACCUMULATED (caller zero-fills)
 *   gb : [cout], accumulated, may be NULL
 * The data gradient is rnc_conv2d_cl_fwd on gy (zero-dilated for stride 2) with the flipped, transposed weights. */
int rnc_conv2d_cl_wgrad(const float* x, int ldx, int cin, const float* gy, int ldg, int cout, int B, int Hin, int Win,
                        int kh, int kw, int stride, float* gw, int ldw, float* gb, void* stream);

/* The same gradient on the tensor cores (tcgen05 kind::tf32, TF32x3 like RNC_CONV_TF32: gy_hi*x_hi + gy_hi*x_lo + gy_lo*x_hi,
 * ~2^-21 per product with fp32's exponent range).  Same arguments and accumulation contract as rnc_conv2d_cl_wgrad, plus:
 *   workspace : rnc_conv2d_umma_wgrad_workspace_bytes(...) bytes of device memory, 16-byte aligned, caller-owned, contents
 *               irrelevant: the TF32 hi/lo planes of x and gy, transposed to channel-major [B][C][H][W'] so that the pixels
 *               (the GEMM's K) are contiguous; the bias gradient is summed by the same pass over gy
 * No TMEM accumulation runs over more than 512 pixels (the tensor core truncates on every accumulate): each chunk is drained
 * into fp32 registers and each work item (co tile, ci tile, tap, pixel range) adds its partial sums with one atomic per element.
 * Returns RNC_ERR_WORKSPACE if workspace_bytes is too small, RNC_ERR_UNSUPPORTED for problems beyond the kernel's index
 * ranges; nothing is launched when an argument is rejected. */
size_t rnc_conv2d_umma_wgrad_workspace_bytes(int cin, int cout, int B, int Hin, int Win, int kh, int kw, int stride);
int rnc_conv2d_umma_wgrad(const float* x, int ldx, int cin, const float* gy, int ldg, int cout, int B, int Hin, int Win,
                          int kh, int kw, int stride, float* gw, int ldw, float* gb,
                          void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RNC_H_ */
