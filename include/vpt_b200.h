/* vpt_b200.h -- C ABI of the B200-native VPT policy forward path (libvpt_b200.so).
 *
 * The reference (openai/Video-Pre-Training) is pure Python on top of torch (it has NO FFI of its own, SURVEY.md
 * section 2.1), so each entry point below replaces the torch / ATen call sequence of one reference site; the
 * reference file:line each one stands in for is cited.  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated otherwise;
 *   - the caller owns every buffer, including workspaces; entry points never allocate device memory, never
 *     synchronise, and enqueue on the given `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, <0 on error; vpt_last_error() returns a thread-local message;
 *   - bf16 tensors are row-major with the channel / feature dimension contiguous (NHWC for images).
 *
 * "row group statistics": several ops take `mr` = float[G][2] = (mean, rstd) of row group g = row / rows_per_group
 * (a frame for GroupNorm(1 group), one token for LayerNorm) and several ops emit `stat_part` = partial
 * (sum, sum of squares) of the values they stored; vpt_stats_finalize turns partials into `mr`.
 */
#ifndef VPT_B200_H_
#define VPT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VPT_OK 0
#define VPT_ERR_ARG (-1)    /* bad argument / unsupported shape */
#define VPT_ERR_CUDA (-2)   /* a CUDA runtime / driver call failed */
#define VPT_ERR_DEVICE (-3) /* a kernel recorded a device-side protocol error (watchdog) */

#define VPT_ABI_VERSION 3

const char* vpt_last_error(void);
int vpt_abi_version(void);
/* Reads and clears the device-side watchdog flag (synchronises the device; for tests / debugging only). */
int vpt_device_error(void);
/* Number of SMs of the current device (grid sizing of the persistent kernels). */
int vpt_num_sms(void);

/* ----------------------------------------------------------------------------------------------------------
 * Tensor-core GEMM / implicit-GEMM 3x3 convolution (tcgen05.mma, TMA-fed, TMEM accumulators).
 *
 *   acc[m][n] = sum_k A[m][k] * B[n][k]                      (bf16 x bf16 -> fp32)
 *   v = a_g * acc - b_g * S1[cls(m)][n] + S2[cls(m)][n]      (a_g,b_g) = (rstd_g, rstd_g*mean_g), or (1,0) if mr==NULL
 *   relu==1: v = max(v,0);  v += residual[m][n];  relu==2: v = max(v,0);  v *= out_scale;  store
 *
 * With conv=0 this is  [LayerNorm ->] Linear [-> ReLU] [+ residual]  of lib/util.py:75-82 (linear flavour),
 * lib/xf.py:336-338,355 (q/k/v/proj), lib/action_head.py:165 and lib/scaled_mse_head.py:35: the LayerNorm is folded
 * (B pre-scaled by gamma; S1[n] = sum_k B[n][k]; S2[n] = sum_k W[n][k]*beta[k] (+ bias[n])).
 * With conv=1 it is  GroupNorm(1) -> Conv2d 3x3 pad 1 -> ReLU [+ residual]  of lib/util.py:75-82 (conv flavour) and
 * lib/impala_cnn.py:50-52: A is the raw NHWC activation tensor [F][H][W][Cin], k = tap*Cin + c, and cls(m) is the
 * border class (row class * 3 + column class, 0 = first, 1 = interior, 2 = last) of output pixel m because the
 * reference zero-pads AFTER normalising.
 * -------------------------------------------------------------------------------------------------------- */
typedef struct vpt_gemm_args {
    const void* A;            /* bf16 */
    const void* B;            /* bf16 [N][K], K contiguous */
    int32_t M, N, K;          /* conv: M = F*H*W, K = 9*Cin */
    int32_t conv;             /* 0 = linear, 1 = 3x3 pad-1 stride-1 convolution */
    int32_t H, W, Cin;        /* conv geometry; Cin % 64 == 0; W*rows == 128 or H*W divides 128 */
    const float* mr;          /* [G][2] (mean, rstd) or NULL */
    int32_t rows_per_group;   /* rows (pixels) per statistics group */
    const float* S1;          /* [ncls][N] (ncls = 9 for conv, 1 for linear) or NULL */
    const float* S2;          /* [ncls][N] or NULL */
    int32_t relu;             /* 0 none, 1 before the residual add, 2 after it */
    float out_scale;
    const void* residual;     /* [M][ld_res] or NULL */
    int32_t residual_f32;     /* 0 = bf16, 1 = fp32 */
    int64_t ld_res;
    void* out;                /* [rows][ld_out] */
    int32_t out_f32;
    int64_t ld_out;
    int32_t seg_len;          /* 0: out row = m; else out row = (m / seg_len) * seg_stride + seg_off + m % seg_len */
    int64_t seg_stride, seg_off;
    float* stat_part;         /* NULL or float2 partials of the stored values (see stat_mode) */
    int32_t stat_mode;        /* 1: [M][P] per row;  2: [ceil(M/32)][P] per 32 rows;  P = vpt_gemm_stat_parts(N) */
    int32_t cluster;          /* CTAs per thread-block cluster sharing the B tile by TMA multicast: 0 = default, 1, 2, 4 */
    /* Column segments (fused projections, e.g. Q | K | V | R of lib/xf.py:334-365 as ONE GEMM over the concatenated weight): columns
     * [dst_n0[i], dst_n0[i+1]) go to dst_out[i] (column 0 of that buffer = column dst_n0[i] of the GEMM) with its own leading dimension
     * and dtype; dst_remap[i] != 0 applies the seg_len / seg_stride / seg_off row remap to that segment only.  ndst == 0: out / ld_out /
     * out_f32 (+ the row remap, if any) describe the single destination.  Every dst_n0[i] must be a multiple of the N tile (256 for
     * N > 256); statistics partials are not supported with segments. */
    int32_t ndst;
    int32_t dst_n0[4];
    void* dst_out[4];
    int64_t dst_ld[4];
    int32_t dst_f32[4];
    int32_t dst_remap[4];
} vpt_gemm_args;

int vpt_gemm_bf16(const vpt_gemm_args* args, void* stream);
/* Cluster size used when vpt_gemm_args.cluster == 0 (tuning knob; 1, 2 or 4; initial value 2). */
int vpt_set_default_cluster(int32_t cluster);
/* Hardware experiment hook used by tools/desc_experiment.py (A rows loaded `shift` rows early, UMMA descriptor start
 * advanced to compensate, base_offset field on/off).  base_offset_mode = -1 (with shift 0) only disables the small-M
 * weight-streaming kernel so that tests can force the tensor-core kernel.  Not for production use. */
int vpt_debug_set(int32_t shift, int32_t base_offset_mode);
/* Number of statistics partials per row (or per 32 rows) the GEMM emits for an N-column output. */
int vpt_gemm_stat_parts(int32_t N);

/* ----------------------------------------------------------------------------------------------------------
 * "ZP" activation layout used by the CNN: bf16 [F][H+1][W+1][C] whose last row (y = H) and last column (x = W) are zero.
 * One shared zero row / column is all the padding a 3x3 pad-1 convolution needs when pixels are addressed linearly
 * (row q = (f*(H+1) + y)*(W+1) + x): the neighbour (dy, dx) of q is row q + dy*(W+1) + dx.  Every producer below writes
 * the zero row / column itself, so the invariant never depends on how the buffer was allocated.
 *
 * GroupNorm(1) -> Conv2d 3x3 pad 1 -> ReLU [+ residual] (lib/util.py:75-82 conv flavour, lib/impala_cnn.py:50-52) on ZP
 * tensors.  Same fold as vpt_gemm_bf16(conv=1) (S1/S2 are [9][Cout] border-class tables), but the input rows are
 * fetched ONCE per 64-channel block and reused by all nine taps from shared memory.
 * -------------------------------------------------------------------------------------------------------- */
typedef struct vpt_conv_zp_args {
    const void* x;            /* bf16 ZP [F][H+1][W+1][Cin] */
    const void* w;            /* bf16 [Cout][9*Cin], k = tap*Cin + c (tap = ky*3 + kx) */
    int32_t F, H, W, Cin, Cout;
    const float* mr;          /* [F][2] (mean, rstd) of x per frame, or NULL */
    const float* S1;          /* [9][Cout] */
    const float* S2;          /* [9][Cout] or NULL */
    int32_t relu;             /* 0 none, 1 before the residual add, 2 after it */
    const void* residual;     /* bf16 ZP [F][H+1][W+1][Cout] or NULL */
    void* out;                /* bf16 ZP [F][H+1][W+1][Cout] */
    float* stat_part;         /* NULL or float2 [F*(H+1)*(W+1)][vpt_conv_zp_stat_parts(Cout)] per-row partials */
    /* Two-norm composition (the post-pool GroupNorm `n` of lib/impala_cnn.py:119 folded into its two consumers instead of running as a
     * pass of its own; tables from vpt_norm2_fold):
     *   Ef        [F][9][Cout] or NULL: per-FRAME additive fold table; out = rstd_f * acc + Ef[f][cls][c] (replaces -rstd*mean*S1 + S2; mr
     *             then carries (0, rstd_f) per frame and S1 / S2 are ignored)
     *   res_scale / res_shift [F][Cout] or NULL: the residual enters as res_scale[f][c] * residual + res_shift[f][c] (the residual
     *             stream x0 = n(y1) recomputed from the un-normalised tensor y1) */
    const float* Ef;
    const float* res_scale;
    const float* res_shift;
} vpt_conv_zp_args;

int vpt_conv3x3_zp(const vpt_conv_zp_args* args, void* stream);
/* SM pairs cooperating on 256-row tiles with tcgen05.mma.cta_group::2 (each CTA stages half of the weight tile):
 * 0 = never, 1 = auto (default: pairs when Cout > 128, where they measure +11-13 %), 2 = always.  Tuning / A-B knob. */
int vpt_set_conv_pair_mode(int32_t on);
/* 1 (default): Cout == 128 layers (of launches with >= 32 tiles) run the operand-swapped kernel (channels as UMMA M, 256 pixels as N; see
 * csrc/conv_zp_t.cuh) with its two-phase epilogue on 16 warps; 0: the regular orientation; 6: the two-phase epilogue on 8 warps; 2 / 4 / 5:
 * timing experiment without an epilogue / fragment epilogue / channel-major single-pass epilogue (DESIGN.md section 4).  Changes
 * vpt_conv_zp_stat_parts(.., 128) and vpt_conv_zp_t_stat_floats.  Tuning / A-B knob: results are identical up to fp32 summation order of the statistics. */
int vpt_set_conv_swap_mode(int32_t on);
int vpt_conv_zp_stat_parts(int32_t F, int32_t H, int32_t W, int32_t Cout);  /* (few frames use narrower weight tiles, hence more partials per row) */
/* Cout == 128 with the operand-swapped kernel's experimental fragment epilogue (vpt_set_conv_swap_mode(4)): its statistics partials are per (tile, warp, frame slot),
 * not per row.  vpt_conv_zp_t_stat_floats > 0 <=> pass a float buffer of that many elements as stat_part and finalise it with
 * vpt_conv_zp_t_stats_finalize (mr[f] = mean, rstd over the H*W*128 interior values of frame f). */
int64_t vpt_conv_zp_t_stat_floats(int32_t F, int32_t H, int32_t W, int32_t Cout);
int vpt_conv_zp_t_stats_finalize(const float* part, float* mr, int32_t F, int32_t H, int32_t W, float eps, void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * Stack-0 first convolution, fused:  u8 -> /255 -> Conv2d(3->C0, 3x3, pad 1) + bias -> ReLU -> max_pool2d(3, 2, 1)
 * (lib/policy.py:39-45, lib/util.py:79-81 with bias, lib/impala_cnn.py:115-117).
 *   img  u8   [F][H][W][3]      w  fp32 [C0][27] ordered (ky, kx, c), already divided by 255
 *   out  bf16 [F][H/2][W/2][C0] (zp=0) or ZP [F][H/2+1][W/2+1][C0] (zp=1)
 *   stat_part float2 [F][vpt_firstconv_stat_parts(F, H, W, C0)]   (H, W multiples of 16; C0 in {64,128,192,256})
 * Two kernels: for W in {32, 64, 128} with H*W <= 16384 the tcgen05 kernel (csrc/firstconv_tc.cuh: operand-swapped implicit GEMM,
 * thread = channel, 3x3/2 max in registers; its partials are per (8 pooled rows, column half, CHANNEL): partial index
 * ((row/8)*2 + half)*C0 + c, so per-channel sums are available to the caller); otherwise the mma.sync kernel (csrc/firstconv.cuh,
 * (H/16)*(W/16) partials per frame).  vpt_set_firstconv_mode(0) forces the mma.sync kernel (A/B knob).
 * out_f32 != 0 (tcgen05 kernel only): `out` is fp32 in the same layout (precision mode, csrc/precise.cuh).
 * -------------------------------------------------------------------------------------------------------- */
int vpt_firstconv_pool(const uint8_t* img, const float* w, const float* bias, void* out, float* stat_part,
                       int32_t F, int32_t H, int32_t W, int32_t C0, int32_t zp, int32_t out_f32, void* stream);
int vpt_firstconv_stat_parts(int32_t F, int32_t H, int32_t W, int32_t C0);
int vpt_set_firstconv_mode(int32_t mode);

/* IDM temporal pre-stage (lib/policy.py:394-403 + :39-45): u8 -> /255 -> Conv3d(3 -> C, kernel (5,1,1), pad (2,0,0)) + bias -> ReLU,
 * per sample over its T frames (zero padded in time at the chunk ends, like the reference's per-sample loop).
 *   img u8 [B][T][H][W][3]   w fp32 [C][15] ordered (dt, c), already divided by 255   out bf16 ZP [B*T][H+1][W+1][C]
 *   stat_part float2 [B*T][vpt_conv3d_stat_parts(H, W, C)] */
int vpt_conv3d_t5(const uint8_t* img, const float* w, const float* bias, void* out, float* stat_part, int32_t B, int32_t T,
                  int32_t H, int32_t W, int32_t C, int32_t out_f32, void* stream);  /* out_f32: fp32 output, same layout (precision mode) */

/* ----------------------------------------------------------------------------------------------------------
 * On-device action codec (csrc/codec.cuh; SURVEY.md row f-3): table look-ups, one thread per action.
 *   vpt_codec_to_env    joint policy action -> MineRL env action: lib/action_mapping.py:215-225 (to_factored, camera-meta nulling) +
 *                       lib/actions.py:154-169 (policy2env; the mu-law camera table cam_lut[nbins] is built by the host with the reference
 *                       formula, lib/actions.py:96-102).  buttons / camera int64 [n]; lut_btn u8 [njoint][20]; lut_cam_off u8 [njoint];
 *                       out [n][22] 8-byte words = 20 int64 button flags + 2 float64 camera angles (ONE device-to-host copy per step);
 *                       *bad counts out-of-range indices.
 *   vpt_codec_from_env  MineRL env action -> joint policy action: lib/actions.py:171-178 (env2policy; the mu-law quantiser :82-94 as
 *                       nbins-1 ascending float64 thresholds) + lib/action_mapping.py:193-213 (from_factored, exclusive groups :65-99,
 *                       inventory override).  buttons int64 [n][20] in lib/actions.py:21-33 order, camera float64 [n][2], strides int64 [9];
 *                       out int64 [n][3] = (buttons index, camera index, is-null-action flag of agent.py:176-180).
 * -------------------------------------------------------------------------------------------------------- */
int vpt_codec_to_env(const int64_t* buttons, const int64_t* camera, const uint8_t* lut_btn, const uint8_t* lut_cam_off, const double* cam_lut,
                     int32_t nbins, int32_t njoint, int64_t n, int64_t* out, int32_t* bad, void* stream);
int vpt_codec_from_env(const int64_t* buttons, const double* camera, const double* thresholds, int32_t nbins, const int64_t* strides,
                       int64_t inventory_idx, int64_t n, int64_t* out, void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * fp32-parity precision mode (csrc/precise.cuh; BASELINE north_star "1e-3 rtol fp32", reference arithmetic lib/xf.py:40,55-63).
 * Contractions stay on vpt_gemm_bf16 (tcgen05): operands split into bf16 hi + lo, three accumulating launches per layer
 * (hi*hi, lo*hi, hi*lo; fp32 output used as the fp32 residual of the next launch).  These entry points are the fp32 glue between
 * them.  All tensors fp32 row-major [rows][C] unless noted.
 *   vpt_group_stats_f32   mr[g] = (mean, rstd) over `per_group` consecutive elements (GroupNorm(1) per frame / LayerNorm per row)
 *   vpt_norm_split_f32    u = [(x - mean_g) * rstd_g] * gamma[c] + beta[c] (mr / gamma / beta optional; group = i / per_group);
 *                         hi = bf16(u), lo = bf16(u - hi) (both or neither) and / or out_f32 = u
 *   vpt_add_f32           out = a + b (b optional), optional ReLU
 *   vpt_maxpool3s2_f32    max_pool2d(3, 2, 1) on NHWC fp32 [F][H][W][C] -> [F][H/2][W/2][C] (lib/impala_cnn.py:117)
 *   vpt_attention_f32     lib/xf.py:18-71 with the mask of lib/masked_attention.py:11-94 and the relative term of lib/xf.py:265-271:
 *                         q [B*t][h], full_k / full_v [B][maxlen+t][h], R [B*t][10*heads] or NULL, b_nd [10][maxlen], first u8 [B][t],
 *                         state_mask u8 [B][maxlen] or NULL (= all False), out [B*t][h]; head_dim 128; causal = clipped_causal mask
 * -------------------------------------------------------------------------------------------------------- */
int vpt_group_stats_f32(const float* x, float* mr, int64_t groups, int64_t per_group, float eps, void* stream);
int vpt_norm_split_f32(const float* x, const float* mr, const float* gamma, const float* beta, void* hi, void* lo, float* out_f32,
                       int64_t n, int32_t C, int64_t per_group, void* stream);
int vpt_add_f32(const float* a, const float* b, float* out, int64_t n, int32_t relu, void* stream);
int vpt_maxpool3s2_f32(const float* in, float* out, int64_t F, int32_t H, int32_t W, int32_t C, void* stream);
int vpt_attention_f32(const float* q, const float* full_k, const float* full_v, const float* R, const float* b_nd, const uint8_t* first,
                      const uint8_t* state_mask, float* out, int32_t B, int32_t t, int32_t maxlen, int32_t heads, int32_t causal,
                      void* stream);
int vpt_conv3d_stat_parts(int32_t H, int32_t W, int32_t C);

/* max_pool2d(kernel 3, stride 2, pad 1) on a non-negative NHWC bf16 tensor (lib/impala_cnn.py:117).
 *   in [F][H][W][C] -> out [F][H/2][W/2][C]   (zp=1: both in the ZP layout, [F][H+1][W+1][C] -> [F][H/2+1][W/2+1][C])
 *   stat_part float2 [F][vpt_pool_stat_parts()] */
int vpt_maxpool3s2(const void* in, void* out, float* stat_part, float* chan_part, int32_t F, int32_t H, int32_t W, int32_t C, int32_t zp,
                   void* stream);  /* chan_part: NULL or float2 [F][P][C] per-channel partials (needs C/8 | 256); with chan_part BOTH partial
                                      buffers hold P = vpt_pool_chan_parts(F, H, W, C) entries per frame instead of vpt_pool_stat_parts */
int vpt_pool_chan_parts(int32_t F, int32_t H, int32_t W, int32_t C);
/* Two-norm composition: the post-pool GroupNorm `n` (lib/impala_cnn.py:119) is not run as a pass; its effect is folded into the two
 * consumers of x0 = n(y1): block 0's conv0 (input y1, weights W*gamma0*gamma_n, per-frame table Ef) and conv1 (residual y1 with a
 * per-frame affine).  From the per-channel (sum, sumsq) partials of y1 [F][NP][C] (vpt_firstconv_pool / vpt_maxpool3s2), gamma_n / beta_n
 * and conv0's class tables Ta = sum W gamma0 beta_n, Tb = sum bf16(W gamma0 gamma_n), Tc = sum W gamma0, Td = sum W beta0 (each [9][Cout],
 * summed over the taps inside the image for the border class and over Cin) this writes, per frame:
 *   mrE [F][2] = (0, rstd0 * rstd1)        Ef [F][9][Cout] = rstd0 Ta - rstd0 rstd1 mu1 Tb - rstd0 mu0 Tc + Td
 *   res_scale [F][C] = rstd1 gamma_n        res_shift [F][C] = beta_n - mu1 rstd1 gamma_n
 * (mu1, rstd1: statistics of y1; mu0, rstd0: statistics of x0, obtained analytically from the per-channel sums). */
int vpt_norm2_fold(const float* chan_part, int32_t NP, int32_t C, int64_t npix, const float* gamma_n, const float* beta_n, const float* Ta,
                   const float* Tb, const float* Tc, const float* Td, int32_t Cout, float eps, float* mrE, float* Ef, float* res_scale,
                   float* res_shift, int64_t F, void* stream);
int vpt_pool_stat_parts(int32_t F, int32_t H, int32_t W, int32_t C);

/* out[m][c] = (in[m][c] - mean_g) * rstd_g * gamma[c] + beta[c],  g = m / rows_per_group   (bf16 in, bf16 out)
 * = nn.GroupNorm(1, C) on NHWC rows (lib/impala_cnn.py:119) and nn.LayerNorm(C) (lib/util.py:195, lib/policy.py:214).
 * Optionally also writes an fp32 copy (out_f32, may be NULL) and emits statistics partials of the bf16 output:
 * stat_part float2 [G][vpt_norm_stat_parts(rows_per_group, C)]. */
int vpt_affine_norm(const void* in, const float* mr, const float* gamma, const float* beta, void* out, float* out_f32,
                    float* stat_part, int64_t M, int32_t C, int32_t rows_per_group, void* stream);
/* The same on ZP tensors [F][H+1][W+1][C], one group per frame: interior pixels are normalised, the zero row / column is
 * rewritten as zero.  stat_part float2 [F][vpt_norm_stat_parts((H+1)*(W+1), C)]. */
int vpt_affine_norm_zp(const void* in, const float* mr, const float* gamma, const float* beta, void* out, float* stat_part,
                       int32_t F, int32_t H, int32_t W, int32_t C, void* stream);
int vpt_norm_stat_parts(int32_t rows_per_group, int32_t C);

/* mr[g] = (mean, rsqrt(var + eps)) from n_per_group float2 partials per group; count = elements per group. */
int vpt_stats_finalize(const float* stat_part, float* mr, int64_t G, int32_t n_per_group, double count, float eps,
                       void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * Transformer-XL style KV memory + banded masked attention with learned relative-position bias
 * (lib/masked_attention.py:11-94,161-178; lib/xf.py:18-71,265-271,334-391; lib/util.py:232-267).
 * -------------------------------------------------------------------------------------------------------- */
/* dst[b][dst_off + r][:] = src[b][src_off + r][:] for r < rows, converting fp32 <-> bf16 (KV memory load / store,
 * lib/xf.py:378-381).  ld = row pitch in elements, *_bstride = batch pitch in elements. */
int vpt_copy_rows(const void* src, int32_t src_f32, int64_t src_bstride, int64_t src_ld, int64_t src_off, void* dst,
                  int32_t dst_f32, int64_t dst_bstride, int64_t dst_ld, int64_t dst_off, int32_t B, int32_t rows,
                  int32_t cols, void* stream);
/* Same for TWO (source, destination) pairs of identical geometry in one launch (the K and the V memory of a layer). */
int vpt_copy_rows2(const void* src, const void* src2, int32_t src_f32, int64_t src_bstride, int64_t src_ld, int64_t src_off, void* dst,
                   void* dst2, int32_t dst_f32, int64_t dst_bstride, int64_t dst_ld, int64_t dst_off, int32_t B, int32_t rows, int32_t cols,
                   void* stream);

/* new_mask[b][j] = j < maxlen - min(t,maxlen) ? (mask[b][j + t] && !first[b]) : 1   (lib/masked_attention.py:86-92)
 * mask_in may be NULL (= all zero, the state after initial_state()).  u8 0/1 arrays. */
int vpt_state_mask_update(const uint8_t* mask_in, const uint8_t* first, int64_t first_stride, uint8_t* mask_out,
                          int32_t B, int32_t t, int32_t maxlen, void* stream);

/*   Q     bf16 [B][t][h]             (h = heads*128, head-major columns, lib/xf.py:96-103)
 *   Kf,Vf bf16 [B][maxlen + t][h]    memory rows then the chunk's rows
 *   R     fp32 [B][t][ld_r]          relative-attention queries, column head*nbasis + n (lib/xf.py:266-267)
 *   b_nd  fp32 [nbasis][maxlen]
 *   first u8 [B] (first[:,0] of the chunk), first_stride = elements between batch rows
 *   smask u8 [B][maxlen] or NULL (all zero)
 *   out   bf16 [B][t][h]
 * logit = q.k / 128 + sum_n R[i][n] b_nd[n][d] over allowed keys, d = maxlen + i - j in [0, maxlen),
 * allowed = j >= maxlen || (!first[b] && smask[b][j]).   causal = 0 selects the IDM variant (mask "none":
 * every chunk key visible, no memory, no relative bias; lib/policy.py:342-392). */
int vpt_attention(const void* Q, const void* Kf, const void* Vf, const float* R, int64_t ld_r, const float* b_nd,
                  const uint8_t* first, int64_t first_stride, const uint8_t* smask, void* out, int32_t B, int32_t t,
                  int32_t maxlen, int32_t heads, int32_t nbasis, int32_t causal, void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * Action heads (lib/action_head.py:163-207)
 * -------------------------------------------------------------------------------------------------------- */
/* out[r][0..n) = log_softmax(in[r][col0 .. col0+n))   in fp32 [rows][ld_in] (already divided by the temperature) */
int vpt_log_softmax(const float* in, int64_t ld_in, int32_t col0, int32_t n, float* out, int64_t rows, void* stream);
/* idx[r] = argmax_j(logits[r][j] - log(-log(u[r][j]))) with u==1 -> 0.999; u == NULL -> plain argmax (deterministic).
 * Ties resolve to the lowest index (torch.argmax). */
int vpt_gumbel_argmax(const float* logits, const float* u, int64_t* idx, int64_t rows, int32_t n, void* stream);
/* lp[r] (+)= logits[r][idx[r]]   (lib/action_head.py:176-184) */
int vpt_gather_logprob(const float* logits, const int64_t* idx, float* lp, int64_t rows, int32_t n, int32_t accumulate,
                       void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * Frame ingest (the step before the path: agent.py:100-103,141-149): bilinear uint8 resize, bit-exact with
 * cv2.resize(..., interpolation=cv2.INTER_LINEAR).  xidx[Wd] / xw[Wd][2] and yidx[Hd] / yw[Hd][2] are the source index and the
 * 11-bit fixed-point weight pairs per destination column / row (computed on the host the way OpenCV does; see agent.py here).
 *   src u8 [F][Hs][Ws][C] -> dst u8 [F][Hd][Wd][C]
 * -------------------------------------------------------------------------------------------------------- */
int vpt_resize_bilinear_u8(const uint8_t* src, uint8_t* dst, const int32_t* xidx, const int16_t* xw, const int32_t* yidx,
                           const int16_t* yw, int32_t F, int32_t Hs, int32_t Ws, int32_t Hd, int32_t Wd, int32_t C, int32_t swap_rb,
                           void* stream);
/* swap_rb != 0 additionally exchanges channels 0 and 2 (cv2.cvtColor(frame, COLOR_BGR2RGB), data_loader.py:116).
 *
 * Cursor overlay of the BC data loader (data_loader.py:34-45,108-115), in place on frames u8 [F][H][W][3]: for every frame with
 * xy[f] = (x, y) >= 0:  frame[y:y+ch, x:x+cw] = uint8(frame * (1 - alpha) + cursor * alpha)  in float64 with numpy's truncation,
 * clipped at the right / bottom border; xy[f].x < 0 = no cursor.  cursor u8 [ch][cw][3], alpha f64 [ch][cw]. */
int vpt_composite_cursor_u8(uint8_t* frames, const uint8_t* cursor, const double* alpha, const int32_t* xy, int32_t F, int32_t H, int32_t W,
                            int32_t ch, int32_t cw, void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * BC step groundwork (behavioural_cloning.py:63-67,119-123): fused torch.optim.Adam(lr, weight_decay) step over ONE flat fp32
 * bucket holding every parameter (gradients in a second flat bucket that data parallelism reduces with a single NCCL
 * all-reduce; grad_scale = 1/world_size).  step counts from 1.  The kernels below fill `grads`.
 * -------------------------------------------------------------------------------------------------------- */
int vpt_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, float grad_scale, int32_t step, void* stream);

/* ----------------------------------------------------------------------------------------------------------
 * BC step backward (behavioural_cloning.py:101-123; the reference gets it from autograd over lib/policy.py).  The host side
 * (video-pre-training_b200/training.py) chains these with the forward entry points above: d(input) of a convolution / linear is
 * vpt_conv3x3_zp / vpt_gemm_bf16 on rotated / transposed weights; the rest is here.  With u = gamma*n + beta, n = (x-mean)*rstd:
 * -------------------------------------------------------------------------------------------------------- */
/* ReLU backward: dz = dout where out > 0, else 0 (bf16, n elements, n % 8 == 0)            lib/util.py:81 */
int vpt_relu_mask(const void* dout, const void* out, void* dz, int64_t n, void* stream);
/* Residual add of the training forward, out = a + b (bf16) per group of `elems_per_group` elements, with float2 (sum, sumsq)
 * partials [groups][vpt_add_stat_parts()] of the stored values (the branch output b is kept separately because its sign
 * pattern is the ReLU mask the backward needs)                                              lib/impala_cnn.py:50-52 */
int vpt_add_stats(const void* a, const void* b, void* out, float* stat_part, int64_t groups, int64_t elems_per_group, void* stream);
int vpt_add_stat_parts(int64_t elems_per_group);
/* Weight-gradient kernel choice: 1 (default) = tap-pairing kernel (csrc/wgrad_tc.cuh: taps whose shifts differ by one row share one
 * activation span and one gradient tile in shared memory, two TMEM accumulators), 0 = one GEMM tile per tap (csrc/gemm_tc.cuh).  A-B knob. */
int vpt_set_wgrad_mode(int32_t mode);
/* 1: forward-path kernels are launched with the programmatic-stream-serialization attribute (programmatic dependent launch): the next
 * kernel is scheduled while the previous one drains and blocks in griddepcontrol.wait until that one has completed and flushed, so only
 * launch latency overlaps.  Default 0 (measured neutral on the rollout CUDA graph; results are bit-identical either way). */
int vpt_set_pdl(int32_t on);
/* Weight gradient on the tcgen05 GEMM (both operands MN-major, K split over CTAs + fixed-order reduction):
 *   out fp32 [M][ntaps*N],  out[m][tap*N + n] = sum_{k in [0,R)} a[k][m] * b[k + shifts[tap]][n]   (rows outside [0,R) are 0)
 * a bf16 [R][lda] = output gradient (M columns), b bf16 [R][ldb] = (normalised) layer input (N columns); no transposes needed.
 * Linear: ntaps = 1, shift 0.  3x3 conv on ZP tensors: ntaps = 9, shifts[tap] = (ky-1)*(W+1) + (kx-1), out is [Cout][tap][Cin].
 * workspace: vpt_wgrad_workspace_bytes() bytes (0 when no K split is used). */
int vpt_wgrad_bf16(const void* a, int64_t lda, const void* b, int64_t ldb, int32_t M, int32_t N, int64_t R, const int32_t* shifts,
                   int32_t ntaps, float* out, void* workspace, int64_t workspace_bytes, void* stream);
int64_t vpt_wgrad_workspace_bytes(int32_t M, int32_t N, int32_t ntaps, int64_t R);
/* GroupNorm(1) / LayerNorm backward in three passes over du, x bf16 [rows][C] (groups of rows_per_group rows, mr [G][2]):
 *   vpt_group_sums     ms[g] = (mean gamma*du, mean gamma*du*n) over the group (`count` real elements; part: [G][parts] float2)
 *   vpt_col_sums       out fp32 [2][C] = (sum_rows du*n, sum_rows du) = (d gamma, d beta); x == NULL: row 1 only (bias gradients);
 *                      workspace [vpt_col_sums_parts()][2][C] floats
 *   vpt_norm_bwd_apply dx = rstd * (gamma*du - ms.x - n*ms.y) [+ add]; zpC > 0: every group is a ZP frame [(zpH+1)(zpW+1)][zpC]
 *                      and its pad row / column is written as zero; relu_x != 0: x is a ReLU output, dx is zeroed where x == 0
 *                      (the ReLU backward of the producer, fused)                          lib/util.py:44-63 (norm placement) */
int vpt_group_sums(const void* du, const void* x, const float* mr, const float* gamma, float* part, float* ms, int64_t rows, int32_t C,
                   int32_t rows_per_group, double count, void* stream);
int vpt_group_sums_parts(int32_t rows_per_group, int32_t C);
int vpt_col_sums(const void* du, int64_t ld_du, const void* x, const float* mr, int64_t rows, int32_t C, int32_t rows_per_group, float* out,
                 float* workspace, void* stream);
int vpt_col_sums_parts(int64_t rows, int32_t C);
/* vpt_col_sums + vpt_group_sums in ONE pass over (du, x) for groups of many rows (GroupNorm frames): the per-channel partials of a
 * slab that lies inside one group also give that group's sums.  out fp32 [2][C], ms fp32 [G][2]; workspace: vpt_norm_sums_workspace()
 * floats. */
int vpt_norm_sums(const void* du, const void* x, const float* mr, const float* gamma, int64_t rows, int32_t C, int32_t rows_per_group,
                  double count, float* out, float* ms, float* workspace, void* stream);
int64_t vpt_norm_sums_workspace(int64_t rows, int32_t C, int32_t rows_per_group);
int vpt_norm_bwd_apply(const void* du, const void* x, const float* mr, const float* gamma, const float* ms, const void* add, void* dx,
                       int64_t rows, int32_t C, int32_t rows_per_group, int32_t zpH, int32_t zpW, int32_t zpC, int32_t relu_x, void* stream);
/* Backward of ReLU -> max_pool2d(3, 2, 1) on ZP tensors (H, W = pool input size): dx[F][H+1][W+1][C] from dy [F][H/2+1][W/2+1][C] and the
 * post-ReLU pool input x; the first maximum in window scan order takes the gradient (torch semantics), windows whose maximum is 0
 * pass none.  workspace: F*(H/2)*(W/2)*C bytes (arg-max position per pooled element)             lib/impala_cnn.py:115-117 */
int vpt_maxpool3s2_bwd(const void* dy, const void* x, void* dx, void* workspace, int32_t F, int32_t H, int32_t W, int32_t C, void* stream);
/* Weight / bias gradient of vpt_firstconv_pool (recomputes the pre-pool map): dW fp32 [C0][27] (same (ky,kx,c) order and /255 scale
 * as w), db [C0]; dy bf16 ZP [F][H/2+1][W/2+1][C0]; workspace [vpt_firstconv_bwd_parts()][C0][28] floats */
int vpt_firstconv_bwd(const uint8_t* img, const float* w, const float* bias, const void* dy, float* dW, float* db, float* workspace, int64_t F,
                      int32_t H, int32_t W, int32_t C0, void* stream);
int vpt_firstconv_bwd_parts(int64_t F, int32_t H, int32_t W);
/* Backward of vpt_attention (causal policy attention): given dO bf16 [B*t][h] writes d q | d k | d v | d R side by side into
 * out bf16 [B*t][ld_out] at columns 0 | h | 2h | 3h (chunk rows only -- the KV memory is detached state,
 * behavioural_cloning.py:111) and d b_nd fp32 [nbasis][maxlen].  workspace: 2*B*heads*t*maxlen floats.   lib/xf.py:18-71,265-271 */
int vpt_attention_bwd(const void* Q, const void* Kf, const void* Vf, const float* R, int64_t ld_r, const float* b_nd, const uint8_t* first,
                      int64_t first_stride, const uint8_t* smask, const void* dO, void* out, int64_t ld_out, float* db_nd, float* workspace,
                      int32_t B, int32_t t, int32_t maxlen, int32_t heads, int32_t nbasis, void* stream);
/* d loss / d logits of a categorical NLL head: out[r][col0 + j] = (exp(logp[r][j]) - [j == idx[r]]) * scale  (bf16)
 *                                                                                          lib/action_head.py:176-184 */
int vpt_softmax_bwd(const float* logp, const int64_t* idx, float scale, void* out, int64_t ld_out, int32_t col0, int64_t rows, int32_t n,
                    void* stream);
/* Loss and gradient of the RL fine-tuning step (training.RLTrainer), one CTA per frame row.  Per head h (nheads <= 4): student
 * log-softmax logp[h] fp32 [rows][n[h]], teacher logp_teacher[h] (logp_teacher == NULL: no teacher, KL term and statistic 0), taken
 * action idx[h] [rows], gradient columns col0[h] of dlog.  Per row: old_logp, adv, ret, vpred fp32 [rows]; mu_rsig fp32 [2] on the
 * device = (mean, 1/std) of the return normaliser.  With lp = sum_h logp[h][a_h], ratio = exp(lp - old_logp), tn = (ret - mean)/std:
 *   dlog[r][col0[h] + j] = inv_temp * (g [j == a_h] + q_j (kl_coef*inv_n (pd_j - pd_t,j - kl_h) + ent_coef*inv_n (pd_j + H_h) - g))  (bf16)
 *   dlog[r][col_v]       = 2 vf_coef inv_n (vpred - tn)                                                                         (bf16)
 * where g = -ratio*adv*inv_n, or 0 where the clipped surrogate is the minimum (ratio > 1+clip_eps with adv > 0, ratio < 1-clip_eps
 * with adv < 0).  stats fp32 [rows][5] = (lp, sum_h kl_h, sum_h H_h, (vpred - tn)^2, clipped flag).
 *                                           lib/action_head.py:176-220, lib/scaled_mse_head.py:37-43, lib/normalize_ewma.py:26-35 */
int vpt_rl_heads_bwd(const float* const* logp, const float* const* logp_teacher, const int64_t* const* idx, const int32_t* n,
                     const int32_t* col0, int32_t nheads, const float* old_logp, const float* adv, const float* ret, const float* vpred,
                     const float* mu_rsig, float clip_eps, float kl_coef, float ent_coef, float vf_coef, float inv_temp, float inv_n,
                     void* dlog, int64_t ld_out, int32_t col_v, float* stats, int64_t rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VPT_B200_H_ */
