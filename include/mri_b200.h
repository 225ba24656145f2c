/*
 * mri_b200.h -- C ABI of libmri_b200.so: the B200 (sm_100a) kernels behind the diffusion hot
 * path of NickB42/mri-image-generation (denoising UNet forward + DDPM q_sample / reverse step).
 *
 * The reference has no FFI layer of its own (SURVEY.md 8b): every FLOP of this path runs inside
 * torch.nn modules.  Each entry point below therefore cites the reference *call site* whose
 * arithmetic it replaces (paths relative to the reference's model_scripts/ directory).
 *
 * Conventions
 *   - plain C types only; device pointers are passed as void* / typed pointers to DEVICE memory
 *     unless the parameter name ends in _host;
 *   - no allocation or free inside any compute call: the caller owns every buffer;
 *   - every compute call takes the CUDA stream (cudaStream_t as void*) it must be enqueued on;
 *   - return value 0 = success, negative = error; mri_last_error() returns a message for the
 *     calling thread's last failure;
 *   - activations are channels-last bf16 (N[D]HWC) inside the path; public tensors of the
 *     reference API (NC[D]HW fp32) are converted at the edges by mri_im2col_* / mri_nhwc_to_nchw.
 */
#ifndef MRI_B200_H
#define MRI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRI_B200_ABI_VERSION 1

int mri_abi_version(void);
const char* mri_last_error(void);
/* 1 if the current device is compute capability 10.x, 0 otherwise, <0 on CUDA error. */
int mri_device_ok(void);

/* ------------------------------------------------------------------------------------------
 * TMA descriptors.  Encodes a CUtensorMap (128 bytes, written to out_map_host) for a tiled
 * view of up to rank 5.  dtype: 0 = bf16, 1 = fp32.  swizzle: 0 none, 1 = 32B, 2 = 64B, 3 = 128B.
 * strides_bytes has rank-1 entries (stride of dims 1..rank-1; dim 0 is contiguous).
 * ------------------------------------------------------------------------------------------ */
int mri_tmap_encode(void* out_map_host, uint64_t global_addr, int dtype, int rank,
                    const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                    int swizzle);

/* ------------------------------------------------------------------------------------------
 * Implicit-GEMM on tcgen05 tensor cores:  D[m, n] = sum_k A[m, k] * B[n, k]  (+ epilogue)
 *
 * Replaces every nn.Conv2d / nn.Conv3d / nn.ConvTranspose2d / nn.ConvTranspose3d call of
 *   slice_cond_2d_ddpm/unet.py:31-32,40,70,89,142,167, ddpm_25d_all_modalities/unet.py (same),
 *   ddpm_3d_ldm/unet_attention.py:34-35,65,72,75,114,123,142,155 (and ddpm_3d_ldm/unet.py),
 * and the two einsums of AttentionBlock3D (unet_attention.py:49-51).
 *
 * One CTA computes a 128 x block_n tile.  Its 128 rows are a box (box[0..3]) of output
 * positions along the four outer dims x1..x4 of the A maps (dim 0 = channels); the K loop
 * walks `n_kb` entries of `ktable`, each naming one 64-channel slab: which A map to read, the
 * channel offset, the (o1..o4) shift of the box (= the filter tap; out-of-bounds rows are
 * zero-filled by TMA, which is the convolution's zero padding) and the K coordinate of the
 * matching 64-wide slab of B (the packed weights).  Stride-2 convolutions and transposed
 * convolutions use parity-view A / output maps, `n_class` > 1 selects per-output-parity tables.
 *
 * ktable entry (8 x int32): { a_map_index, c0, o1, o2, o3, o4, b_k, 0 }.
 * Epilogue: + bias[n] + rowbias[sample, n] + bias_m[x1] + residual tile, optional GroupNorm
 * partial sums (sum, sum of squares per (sample, stats group)) and a TMA store through o_maps.
 * ------------------------------------------------------------------------------------------ */
typedef struct MriGemmArgs {
  const void* a_maps;     /* device: CUtensorMap[], rank-5 bf16, box {64, box[0..3]}, swizzle 128B */
  const void* b_map;      /* device: CUtensorMap, rank-4 bf16 {K, rows, z1, z2}, box {64, block_n,1,1} */
  const void* o_maps;     /* device: CUtensorMap[n_class], rank-5 output, box {chunk, box[0..3]} */
  const int32_t* ktable;  /* device: [n_class][n_kb][8] */
  int32_t n_kb;
  int32_t n_class;
  int32_t tiles[4];       /* number of boxes along x1..x4 */
  int32_t box[4];         /* box extent along x1..x4; product <= 128 */
  int32_t ext[4];         /* valid output extent along x1..x4 (row validity for the statistics) */
  int32_t n_tiles_n;      /* tiles along N */
  int32_t block_n;        /* 16, 32, 64, 128 or 256 */
  int32_t n_total;        /* valid output columns */
  int32_t bz_sel[2];      /* B coords z1, z2: 0 -> 0, 1 -> class, 2..5 -> tile index along x1..x4 */
  int32_t sample_dim;     /* 1..4: which x dim is the sample (batch) index; 0 = none */
  int32_t out_f32;        /* 0: bf16 output, 1: fp32 output */
  const float* bias;      /* [n_total] or NULL */
  const float* bias_m;    /* [ext[0]] bias along x1 (rows) or NULL */
  const float* rowbias;   /* [samples][rowbias_ld] or NULL (time-embedding projection) */
  int32_t rowbias_ld;
  double* stats;          /* [samples][stats_ld][2] (sum, sumsq) accumulated with fp64 atomics
                             (order-insensitive to ~1e-16, i.e. reproducible), or NULL */
  int32_t stats_ld;       /* statistics groups per sample */
  int32_t stats_cpg;      /* channels per statistics group (multiple of 8) */
  int32_t stages;         /* TMA ring depth; 0 = as deep as shared memory allows (4..8) */
  int32_t sched;          /* 0: every tile's K loop stays in one CTA; 1: the tiles that do not fill a
                             whole wave of the persistent grid are split along K across all CTAs
                             ("stream-K", needs the workspace), the rest run as whole tiles */
  const void* r_maps;     /* device: CUtensorMap[n_class] residual tensor (bf16) through the output
                             view, boxes as o_maps, or NULL.  Used when swap_ab = 1 ... */
  const void* r_base;     /* ... and the same residual as a plain pointer (swap_ab = 0): the element
                             added to output (class c, box position x, column n) is
                             r_base[r_cls_off[c] + sum_i x_i * r_stride[i] + n]  (n_class <= 8).
                             Both are set or both NULL. */
  int64_t r_cls_off[8];
  int64_t r_stride[4];
  float* sk_partials;     /* stream-K workspace (mri_gemm_workspace_bytes), shared by all launches */
  int32_t* sk_flags;      /* [sk_ctas] zero-initialised once; the kernel resets what it raises */
  int32_t sk_ctas;
  int32_t swap_ab;        /* 1: weights are the M = 128 MMA operand, two boxes of positions the N = 256
                             operand (needs block_n 128, n_total % 128 == 0, bf16 output) */
  int32_t staging2;       /* set by the library (short K loops: second set of staging buffers) */
  int32_t xreuse;         /* swap_ab only, box[0] == 8 and 16 groups per box: the a_maps boxes are 10
                             positions wide along x1 (x - 1 .. x + 8) and k-table entries form groups
                             (entry[7] = 1 marks a group leader) that share one activation tile; each
                             entry's o1 in {-1, 0, 1} selects the view of that tile (3 taps per load).
                             2: box[1] == 16 as well, tiles are 10 x 18 and the nine (o2, o1) taps
                             share one (correct, but slower on B200: see plan.conv_plan) */
  int32_t tile_fast_dim;  /* 0..3: the x dim along which consecutive boxes (and the two boxes of a
                             swap_ab tile) advance first.  0 = x1.  3-D stride-1 convolutions use 2
                             (depth): a CTA then walks a column of boxes plane by plane, so the input
                             planes shared by the kd = -1, 0, +1 taps of neighbouring tiles are still
                             in L2 (measured: DRAM reads of a top-level cfg4 conv 3.1x -> ~1x input) */
  uint64_t* trace;        /* profiling only (normally NULL): [grid][16] per-CTA timestamps / wait cycles, see gemm_tc.cu */
} MriGemmArgs;

/* dynamic shared memory one CTA uses for (block_n, swap_ab, requested stages; 0 = maximum) */
int mri_gemm_smem_bytes(int block_n, int swap_ab, int stages);
/* bytes of the stream-K workspace for the current device: [n_ctas][128][256] fp32 partial tiles
 * followed by 1 KB holding int32 flags[n_ctas] (the caller zeroes the flags once). */
int mri_gemm_workspace_bytes(int* n_ctas_out);
int mri_gemm_launch(const MriGemmArgs* args_host, void* stream);

/* ------------------------------------------------------------------------------------------
 * GroupNorm (+SiLU, + time-embedding add, + residual add), channels-last bf16.
 * Replaces nn.GroupNorm + nn.SiLU + the broadcast adds of
 *   slice_cond_2d_ddpm/unet.py:43-56,194-197 (post-norm: h = silu(gn(h)); h += silu(lin(t));
 *   return h + res), ddpm_3d_ldm/unet_attention.py:38,79-85,199 (pre-norm).
 * x, y: [samples][spatial][C] bf16.  stats: fp64 [samples][stats_ld][2] (sum, sumsq) over fine groups
 * of stats_cpg channels starting at group index stats_g0; `groups` normalisation groups of
 * C/groups channels each are formed by summing adjacent fine groups.
 * y = act(gn(x)*gamma+beta) + rowbias[sample][c] + residual ;  act = SiLU if silu != 0.
 * ------------------------------------------------------------------------------------------ */
int mri_gn_stats(const void* x, double* stats, int samples, int64_t spatial, int C, int stats_ld,
                 int stats_g0, int stats_cpg, void* stream);
int mri_gn_apply(const void* x, void* y, const double* stats, const float* gamma,
                 const float* beta, const float* rowbias, int rowbias_ld, const void* residual,
                 int samples, int64_t spatial, int C, int groups, int stats_ld, int stats_g0,
                 int stats_cpg, float eps, int silu, void* stream);

/* ------------------------------------------------------------------------------------------
 * Time / slice-position embedding path (tiny GEMMs, fp32).
 * mri_sinusoidal: SinusoidalPosEmb.forward, slice_cond_2d_ddpm/unet.py:12-25 (identical copies
 *   in ddpm_25d_all_modalities/unet.py:13-26, ddpm_3d_ldm/unet.py:12-25, unet_attention.py:12-25).
 *   freqs[dim/2] = exp(arange(dim/2) * -(ln 1e4 / (dim/2 - 1))) in fp32, built on the host.
 * mri_linear: y[b,o] = act(bias[o] + sum_i x[b,i] W[o,i]) (+ addend[b,o]); act: 0 none, 1 SiLU.
 *   nn.Linear sites: unet.py:124-136 (time_mlp, slice_mlp), :34,48-49 (per-block projection, SiLU
 *   applied to the projection in 2D), unet_attention.py:68,81-83 (no SiLU in 3D).
 * ------------------------------------------------------------------------------------------ */
int mri_sinusoidal(const int64_t* t, const float* freqs, float* out, int batch, int dim,
                   void* stream);
int mri_linear(const float* x, const float* W, const float* bias, const float* addend, float* y,
               int batch, int in_f, int out_f, int act, void* stream);

/* ------------------------------------------------------------------------------------------
 * Layout edges.
 * mri_im2col: explicit patch matrix for the thin-channel first convolution (Cin = 1, 3, 20):
 *   src is NC[D]HW fp32 (src_f32=1) ; dst [samples*D*H*W][kpad] bf16 with column
 *   ((kd*kh_+kh)*kw_+kw)*cin + c, zero padded to kpad.  `ksize` cubic/square kernel, pad = ksize/2.
 *   A second source (src2, cin2 channels, may be NULL) is concatenated on channels
 *   (ddpm_25d_all_modalities/unet.py:198-199).
 * mri_nhwc_to_nchw: dst[n][c][s] fp32 = src[n][s][c] bf16 for c < C (src row pitch ldc).
 * mri_nchw_to_nhwc: dst[n][s][c] bf16 = src[n][c][s] fp32.
 * ------------------------------------------------------------------------------------------ */
int mri_im2col(const float* src, const float* src2, void* dst, int samples, int cin, int cin2,
               int D, int H, int W, int ksize, int ndim, int kpad, void* stream);
/* Weight re-pack after a parameter update (torch.optim step, ddpm_3d_ldm/train.py:399): every
 * packed buffer of a program is a gather of fp32 parameter elements.  One launch refreshes all
 * segments: dst[i] = idx[i] < 0 ? 0 : src[idx[i] >> 28][idx[i] & 0x0fffffff], converted to bf16
 * when dst_bf16.  block0 = index of the segment's first 2048-element block (prefix sum, the host
 * passes the total).  segs_dev lives in device memory. */
typedef struct MriGatherSeg {
  void* dst;
  const int32_t* idx;
  const float* src[4];
  int64_t n;
  int64_t block0;
  int32_t dst_bf16;
  int32_t reserved;
} MriGatherSeg;
int mri_gather_pack(const MriGatherSeg* segs_dev, int n_segs, int64_t total_blocks, void* stream);

/* Thin-Cout convolution (out_conv: 128 -> 3 / 64 -> 1 / 64 -> 4 channels,
 * slice_cond_2d_ddpm/unet.py:167, unet_attention.py:155) finished from the per-tap products
 * Y[q][tap*cout + co] = W[tap][co] . x[q] (one tensor-core GEMM, K = Cin):
 *   out[o][co] = bias[co] + sum_tap Y[o + tap - ksize/2][tap*cout + co]   (zero outside the volume)
 * y: [samples][D][H][W][ldy] bf16, out: [samples][D][H][W][ldo] bf16 (channels >= cout written 0). */
int mri_tap_gather(const void* y, void* out, const float* bias, int samples, int D, int H, int W,
                   int ksize, int ndim, int cout, int ldy, int ldo, void* stream);
/* mri_im2col4: the same patch matrix from a channels-last bf16 copy of the input, src
 * [samples][D*H*W][cp] with cp = channels padded to a multiple of 4 (mri_nchw_to_nhwc writes it):
 * dst[m][tap*cp + c], zero padded to kpad.  The packed weights use the same (tap, padded channel)
 * column order. */
int mri_im2col4(const void* src, void* dst, int samples, int cp, int D, int H, int W, int ksize,
                int ndim, int kpad, void* stream);
int mri_nhwc_to_nchw(const void* src, float* dst, int samples, int64_t spatial, int C, int ldc,
                     void* stream);
int mri_nchw_to_nhwc(const float* src, void* dst, int samples, int64_t spatial, int C, int ldc,
                     void* stream);

/* First convolution of the UNets for inference (in_conv / init_conv with 1..4 input channels, 3^ndim
 * taps, padding 1: ddpm_3d_ldm/unet_attention.py:114,161; slice_cond_2d_ddpm/unet.py:137,185) as ONE
 * tcgen05 kernel that builds the patch matrix in shared memory from the fp32 NC[D]HW input
 * (csrc/thin_conv.cu): y bf16 [samples][D*H*W][cout] = conv(x) + bias, plus the GroupNorm(8, cout)
 * partial sums (sum, sum of squares per (sample, group), fp64 [samples][stats_ld][2], ADDED to --
 * zero them first) when stats != NULL.  w_packed: bf16 [cout][128], column = tap * 4 + channel with
 * taps in (kd, kh, kw) order, zero padded.  cout must be 64 or 128. */
int mri_thin_in_conv(const float* x, const void* w_packed, const float* bias, void* y, double* stats,
                     int stats_ld, int samples, int cin, int D, int H, int W, int ndim, int cout,
                     void* stream);

/* Strided 4-D copy with dtype conversion, dst[i0,i1,i2,i3] = (dst_dtype) src[i0,i1,i2,i3] with
 * element strides src_strides / dst_strides (host int64[4]) and `shape` (host int64[4]); dtypes
 * 0 = bf16, 1 = f32, 2 = f64 (source only).  Used for the few layout shuffles of the backward
 * launch list that torch's autograd does with copy_/permute (e.g. the per-head attention
 * gradients back into the qkv layout, unet_attention.py:44-47), so that no ATen kernel runs
 * inside a replayed step.  mri_memset_zero: cudaMemsetAsync(ptr, 0, bytes) on `stream`. */
int mri_copy_cast(const void* src, int src_dtype, const int64_t* src_strides, void* dst,
                  int dst_dtype, const int64_t* dst_strides, const int64_t* shape, void* stream);
int mri_memset_zero(void* ptr, int64_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused bottleneck attention, inference (AttentionBlock3D.forward, ddpm_3d_ldm/unet_attention.py:
 * 44-52: q, k, v = qkv.chunk(3); attn = softmax(einsum('bhcn,bhcm->bhnm') * d^-0.5); out =
 * einsum('bhnm,bhcm->bhcn')): O = softmax(Q K^T * scale) V per (sample, head) in ONE kernel --
 * tcgen05 MMAs with S and O in TMEM, online softmax between them, logits and probabilities never
 * written to HBM (csrc/attn_flash.cu).
 *   qk_map: CUtensorMap over the token-major qkv tensor, bf16, dims {row length, n, batch}, box
 *           {64, 128, 1}, 128B swizzle; head h reads q at columns [h*d, (h+1)*d) and k at
 *           [k_col0 + h*d, ...).
 *   vt_map: CUtensorMap over v^T, bf16, dims {npad (keys, contiguous), rows, batch}, box
 *           {64, d, 1}, 128B swizzle; head h reads rows [v_row0 + h*d, ...).  Keys >= n must be
 *           outside the tensor or zero.
 *   out:    bf16 [batch][n][ld_out]; head h writes columns [h*d, (h+1)*d).
 * d must be 64 or 128 (mri_attn_flash_supported).  Training keeps the unfused GEMM / softmax
 * launches: its backward pass needs the probabilities.
 * ------------------------------------------------------------------------------------------ */
typedef struct MriAttnArgs {
  const void* qk_map;
  const void* vt_map;
  void* out;
  int32_t batch, heads, n, d;
  int32_t C;        /* heads * d */
  int32_t k_col0, v_row0, ld_out;
  float scale;      /* d^-0.5 */
  int32_t reserved;
} MriAttnArgs;
int mri_attn_flash_supported(int d);
int mri_attn_flash_launch(const MriAttnArgs* args, void* stream);

/* Row softmax for the bottleneck attention (unet_attention.py:50): P = softmax(S * scale),
 * S fp32 [rows][ld_s], P bf16 [rows][ld_p], `cols` valid columns (padding columns written 0). */
int mri_softmax_rows(const float* S, void* P, int64_t rows, int cols, int ld_s, int ld_p,
                     float scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * DDPM arithmetic, fp32, bit-exact w.r.t. the reference's eager association order.
 * All take x as [samples][per_sample] fp32 (NC[D]HW flattened) and t as int64[samples].
 *
 * mri_q_sample:  out = sqrt_ac[t]*x0 + sqrt_1mac[t]*noise
 *   (slice_cond_2d_ddpm/diffusion.py:60-75, ddpm_25d_all_modalities/diffusion.py:59-74,
 *    ddpm_3d_ldm/diffusion.py:68-82)
 * mri_ddpm_step: out = c1[t]*(x - (beta[t]/s[t])*eps) + ((t!=0) * sqrt(pv[t])) * noise
 *   (p_sample: slice_cond_2d_ddpm/diffusion.py:115-132, ddpm_25d.../diffusion.py:96-112,
 *    ddpm_3d_ldm/diffusion.py:106-126).  eps is either fp32 in x's layout (eps_nhwc_ldc = 0) or
 *    the bf16 channels-last UNet output with row pitch eps_nhwc_ldc and `channels` channels.
 * mri_ddim_step: x0=(x-sqrt(1-a_t)*eps)/max(sqrt(a_t),1e-8); out=sqrt(a_p)*x0+sqrt(1-a_p)*eps
 *   (ddpm_3d_ldm/diffusion.py:168-186)
 * mri_minsnr_loss: per-sample mean((pred-noise)^2) weighted by min(snr[t],gamma)/snr[t], mean
 *   over samples (ddpm_3d_ldm/diffusion.py:91-99); gamma <= 0 means plain MSE (F.mse_loss,
 *   ddpm_25d_all_modalities/diffusion.py:89).  loss_out: float[1]; per_sample: float[samples].
 * ------------------------------------------------------------------------------------------ */
int mri_q_sample(const float* x0, const float* noise, const int64_t* t, const float* sqrt_ac,
                 const float* sqrt_1mac, float* out, int samples, int64_t per_sample, void* stream);
int mri_ddpm_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                  const float* noise, const int64_t* t, const float* betas, const float* sqrt_1mac,
                  const float* sqrt_recip_alphas, const float* post_var, float* out, int samples,
                  int64_t per_sample, void* stream);
int mri_ddim_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                  const int64_t* t, const int64_t* t_prev, const float* alphas_cumprod, float* out,
                  int samples, int64_t per_sample, void* stream);
/* mri_dpmpp_step: one DPM-Solver++(2M) step (not in the reference).  coef: device fp32 [rows][5]
 * table of (s, r, A, B, C) rows (schedules.dpmpp_2m_table); k: device int64 row index (nullptr:
 * row 0).  With that row, per element:
 *     x0 = (x - s*eps)*r ;  out = (A*x + B*x0) + C*(x0 - x0_prev) ;  x0_prev = x0
 * fp32, that association, no FMA contraction; the C term is not evaluated when C == 0, so
 * x0_prev is not read on a first-order row (it may hold NaN there).  x0_prev is fp32 in x's
 * layout; eps as for mri_ddim_step (ldc >= channels).  x and out may alias. */
int mri_dpmpp_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                   float* x0_prev, const float* coef, const int64_t* k, float* out, int samples,
                   int64_t per_sample, void* stream);
/* mri_step_table_advance: k[0] += 1, then t[b] = ts[min(k[0], rows - 1)] for b < n, in one
 * launch (race-free for any n) -- the bookkeeping between two replays of a DPM-Solver++ step. */
int mri_step_table_advance(int64_t* t, int n, int64_t* k, const int64_t* ts, int rows, void* stream);
/* mri_inpaint_merge: inpainting by replacement (not in the reference), in place per element:
 *     x = mask ? x : (tau < 0 ? known : sqrt_ac[tau]*known + sqrt_1mac[tau]*z),  tau = t[n] + t_delta
 * with mri_q_sample's operations.  mask: one uint8 per element (nonzero = regenerate), known fp32,
 * both in x's layout.  z comes from `noise` (fp32, x's layout) or, with rng, from Philox under the
 * ATen mapping at generator offset rng[1] + rng_skip (rng_skip a multiple of 4): the
 * torch.randn_like that follows a draw which advanced the offset by rng_skip.  Exactly one of
 * noise / rng.  Values of known where mask != 0 and of x where mask == 0 never reach the output
 * (selected, not blended: NaN there is harmless); both buffers must still be readable in full. */
int mri_inpaint_merge(float* x, const float* known, const uint8_t* mask, const float* noise,
                      const uint64_t* rng, uint64_t rng_skip, const int64_t* t, int64_t t_delta,
                      const float* sqrt_ac, const float* sqrt_1mac, int samples, int64_t per_sample,
                      void* stream);
/* mri_kspace_work_bytes: the size of mri_kspace_merge's work buffer, samples * channels * H *
 * (W / 2 + 1) complex fp32 values.  H and W must be at most 512. */
int mri_kspace_work_bytes(int samples, int channels, int H, int W, size_t* bytes_out);
/* mri_kspace_merge: k-space data consistency (not in the reference; Song et al., ICLR 2022), in
 * place on x (fp32, NCHW, samples x channels planes of H x W), per sample with tau = t[n] + t_delta:
 *     x = x - P(x - sqrt_1mac[tau]*z) + sqrt_ac[tau]*x_zf        (tau >= 0)
 *     x = x - P x + x_zf                                          (tau < 0; z is not used)
 * P u = Re F^-1(M . F u), F the orthonormal unshifted 2-D DFT of each plane, M = kmask (one uint8
 * per element of x, nonzero = measured).  kmask MUST be Hermitian-symmetric, M(k) = M(-k): the
 * kernel forms only the half spectrum (W / 2 + 1 columns), so P is then the orthogonal projector
 * P = P^T = P^2; the host completes a measured mask before the call.  x_zf: fp32 in x's layout.
 * z as for mri_inpaint_merge: `noise`, or with rng the Philox draw at offset rng[1] + rng_skip.
 * Exactly one of noise / rng.  work: caller-owned, at least mri_kspace_work_bytes, 8-byte aligned.
 * Three launches (row DFT, column DFT + mask + inverse column DFT, inverse row DFT + update), each
 * a direct fp32 summation against an exactly indexed sincospi twiddle table: O(HW(H + W)) per
 * plane, relative error near fp32 rounding.  H and W at most 512. */
int mri_kspace_merge(float* x, const float* x_zf, const uint8_t* kmask, const float* noise,
                     const uint64_t* rng, uint64_t rng_skip, const int64_t* t, int64_t t_delta,
                     const float* sqrt_ac, const float* sqrt_1mac, void* work, size_t work_bytes,
                     int samples, int channels, int H, int W, void* stream);
/* mri_kspace3d_work_bytes: the size of mri_dc_project3d's work buffer: samples * channels * D * H *
 * (W / 2 + 1) complex fp32 values (rounded up to 256 bytes), then one fp64 partial sum per 16 rows
 * of every (sample, channel) volume.  D, H and W must be at most 512. */
int mri_kspace3d_work_bytes(int samples, int channels, int D, int H, int W, size_t* bytes_out);
/* mri_dc_project3d: the k-space data term of measurement-guided sampling (not in the reference),
 * per (sample, channel) volume of u (fp32 NCDHW, D x H x W):
 *     g = Re F^-1(M . F u) - x_zf,        gg[n] = sum over sample n of g^2   (fp32 out)
 * F the orthonormal unshifted 3-D DFT over (D, H, W), M = kmask (one uint8 per element of u,
 * nonzero = measured) and MUST be Hermitian-symmetric, M(k) = M(-k): only the half spectrum
 * (W / 2 + 1 bins) is formed, as in mri_kspace_merge.  x_zf, g: fp32 in u's layout.  Five DFT
 * launches (rows, forward H, forward D . M . inverse D, inverse H, inverse rows + g), each a direct
 * fp32 summation against an exactly indexed sincospi twiddle table (the sums of mri_kspace_merge),
 * and one reduction: gg is summed in fp64 in a fixed order, so two launches are bit-identical.
 * work: caller-owned, at least mri_kspace3d_work_bytes, 8-byte aligned.  D, H, W at most 512. */
int mri_dc_project3d(const float* u, const float* x_zf, const uint8_t* kmask, float* g, float* gg,
                     void* work, size_t work_bytes, int samples, int channels, int D, int H, int W,
                     void* stream);
/* mri_dc_mask: the image-space data term of measurement-guided sampling (not in the reference):
 *     g = mask ? 0 : u - known,           gg[n] = sum over sample n of g^2   (fp32 out)
 * mask: one uint8 per element, nonzero = regenerate (known is not read there), 0 = keep; u, known,
 * g fp32 of samples * per_sample elements.  gg is summed in fp64 in a fixed order.  work: at least
 * 1024 bytes per sample, 8-byte aligned.  At most 65535 samples. */
int mri_dc_mask(const float* u, const float* known, const uint8_t* mask, float* g, float* gg, void* work,
                size_t work_bytes, int samples, int64_t per_sample, void* stream);
/* mri_guided_x0: the clean estimate of a guided step, divided by the latent scale (not in the
 * reference), per element with ts = t[n]:
 *     out = (z - sqrt_1mac[ts]*eps) / sqrt_ac[ts] * inv_s[0]
 * fp32 with round-to-nearest in that order.  eps as the step ops read it: fp32 in z's layout
 * (eps_nhwc_ldc = 0) or the bf16 channels-last UNet output [n][spatial][ldc].  inv_s: one device
 * fp32 value (1 / latent scale). */
int mri_guided_x0(const float* z, const void* eps, int eps_nhwc_ldc, int channels, const int64_t* t,
                  const float* sqrt_ac, const float* sqrt_1mac, const float* inv_s, float* out,
                  int samples, int64_t per_sample, void* stream);
/* mri_guided_eps: the guided noise prediction (not in the reference; DPS's normalisation, Chung et
 * al. ICLR 2023, applied to the clean estimate as MPGD, He et al. ICLR 2024), per element with
 * ts = t[n] and c = lam[0] / sqrt(gg[n]) (c = 0 when gg[n] = 0):
 *     delta = -c * (dz * inv_s[0]),   out = eps - (sqrt_ac[ts] / sqrt_1mac[ts]) * delta
 * and out = eps exactly where c = 0.  dz: the decoder's input gradient D^T g (fp32 in out's
 * layout), gg: mri_dc_project3d's / mri_dc_mask's sums, lam / inv_s: one device fp32 value each.
 * eps as for mri_guided_x0; out: fp32 NCDHW, the eps an unchanged reverse-step update then reads. */
int mri_guided_eps(const void* eps, int eps_nhwc_ldc, int channels, const float* dz, const float* gg,
                   const float* lam, const float* inv_s, const int64_t* t, const float* sqrt_ac,
                   const float* sqrt_1mac, float* out, int samples, int64_t per_sample, void* stream);
/* mri_repaint_undo: RePaint's undo step (not in the reference), in place per element with
 * l = t[n] in [-1, T - 2] per sample:
 *     x = sqrt(alphas[l + 1])*x + sqrt(betas[l + 1])*z
 * fp32, two multiplies and one add rounded to nearest (no FMA contraction), sqrt rounded to
 * nearest: bit-identical to eager alphas[l + 1].sqrt() * x + betas[l + 1].sqrt() * z.  z as for
 * mri_inpaint_merge: `noise`, or with rng the Philox draw at offset rng[1] + rng_skip.  Exactly
 * one of noise / rng. */
int mri_repaint_undo(float* x, const float* noise, const uint64_t* rng, uint64_t rng_skip,
                     const int64_t* t, const float* alphas, const float* betas, int samples,
                     int64_t per_sample, void* stream);
/* mri_vb_terms: the per-sample sums of one evaluation step of the variational bound (not in the
 * reference), at l = t[n] in [0, timesteps - 1] per sample (other values add nothing), for
 * x_t = q_sample(x0, l, z) and the model's eps:
 *     acc[n][l][0] += sum (eps - z)^2
 *     l = 0:  acc[n][0][1] += sum -log p(x0 | x_t),  prior[n] += sum x0^2  (prior nullable)
 * p(x0 | x_t) has the mean of mri_ddpm_step at t = 0 and log-scale 0.5 * post_log_var[0];
 * decoder 0: discretized Gaussian over 8-bit bins of [-1, 1] (improved-diffusion's
 * discretized_gaussian_log_likelihood), 1: Gaussian density (continuous data; may be negative).
 * x0, x_t, z: fp32 [samples][per_sample]; eps as for mri_ddim_step (ldc >= channels).  acc: fp64
 * [samples][timesteps][2], prior: fp64 [samples], both accumulated into.  fp32 per element, fp64
 * partial sums with one atomicAdd per block, sample and quantity.  samples <= 65535. */
int mri_vb_terms(const float* x0, const float* x_t, const void* eps, int eps_nhwc_ldc, int channels,
                 const float* z, const int64_t* t, const float* betas, const float* sqrt_1mac,
                 const float* sqrt_recip_alphas, const float* post_var, const float* post_log_var,
                 int decoder, double* acc, double* prior, int timesteps, int samples,
                 int64_t per_sample, void* stream);
int mri_minsnr_loss(const float* pred, const float* noise, const int64_t* t, const float* snr,
                    float gamma, float* per_sample_out, float* loss_out, int samples,
                    int64_t per_sample, void* stream);
/* t[i] += delta for i < n (advances the device-resident timestep inside a CUDA graph) */
int mri_add_i64(int64_t* t, int n, int64_t delta, void* stream);

/* ------------------------------------------------------------------------------------------
 * In-kernel Philox4x32-10 + Box-Muller noise, bit-identical to torch.randn / torch.randn_like on
 * the same device for the same generator state -- the draws the reference makes at
 * ddpm_3d_ldm/diffusion.py:75,86,122,131 and slice_cond_2d_ddpm/diffusion.py:67,93,129,140
 * (ATen mapping: element e of a tensor of `numel` elements is component (e % (4 Tt)) / Tt of the
 * curand_normal4 call number e / (4 Tt) of subsequence e % Tt, Tt = 256 * min(#SM *
 * (maxThreadsPerSM / 256), ceil(numel / 256)); ATen/native/cuda/DistributionTemplates.h).
 * `rng`: device uint64[2] = {seed, philox offset} -- what torch.cuda's generator reports through
 * initial_seed() / get_offset(); the offset must be a multiple of 4.  One draw of `numel` normals
 * advances the offset by mri_randn_offset_increment(numel) (host helper, no launch).
 *   mri_randn:          out[e] = z[e]
 *   mri_q_sample_rng:   out = sqrt_ac[t]*x0 + sqrt_1mac[t]*z, noise_out = z (nullable)
 *   mri_ddpm_step_rng:  mri_ddpm_step with z drawn in the kernel (x and out may alias)
 *   mri_step_advance:   t[i] += delta (and t_prev[i] = max(t_prev[i] + delta, 0), nullable) for
 *                       i < n; rng[1] += rng_increment
 *                       (rng nullable) -- the bookkeeping between two replays of a captured step
 * ------------------------------------------------------------------------------------------ */
/* mri_rng_seed: rng[0] = seed, rng[1] = offset, stream-ordered (no host synchronisation) */
int mri_rng_seed(uint64_t* rng, uint64_t seed, uint64_t offset, void* stream);
/* mri_tap_gather_step: the thin output convolution finished INSIDE the reverse step
 * (ddpm_3d_ldm/unet_attention.py:155,199 out_conv -> diffusion.py:118-126 / 168-186).  Y is the
 * "GEMM over all taps" of out_conv (see mri_tap_gather): eps[q][co] = bias[co] + sum over taps of
 * Y[q + off(tap)][tap * cout + co], rounded to bf16 exactly as mri_tap_gather stores it, and
 *   mode 0: x <- DDPM update with z drawn in the kernel (ATen mapping over the whole state tensor),
 *   mode 1: x <- DDIM update (t_prev, alphas_cumprod),
 *   mode 2: eps only (eps_out bf16 [positions][ldo] required; otherwise optional),
 *   mode 3: x <- DPM-Solver++(2M) update of mri_dpmpp_step (x0_prev, coef, k; bf16-rounded eps).
 * x is the fp32 NC[D]HW sampler state [samples][cout][D][H][W], updated in place; 3^ndim taps,
 * ndim 2 (D = 1) or 3, cout 1..4.  The predicted noise never goes to HBM in modes 0 / 1 / 3.
 * Arguments a mode does not use may be null. */
int mri_tap_gather_step(const void* y, const float* bias, int samples, int D, int H, int W, int ndim,
                        int cout, int ldy, float* x, void* eps_out, int ldo, int mode,
                        const uint64_t* rng, const int64_t* t, const int64_t* t_prev,
                        const float* betas, const float* sqrt_1mac, const float* sqrt_recip_alphas,
                        const float* post_var, const float* alphas_cumprod, float* x0_prev,
                        const float* coef, const int64_t* k, void* stream);
int mri_randn_offset_increment(int64_t numel, uint64_t* increment_out);
int mri_randn(float* out, int64_t numel, const uint64_t* rng, void* stream);
int mri_q_sample_rng(const float* x0, const uint64_t* rng, const int64_t* t, const float* sqrt_ac,
                     const float* sqrt_1mac, float* out, float* noise_out, int samples,
                     int64_t per_sample, void* stream);
int mri_ddpm_step_rng(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                      const uint64_t* rng, const int64_t* t, const float* betas,
                      const float* sqrt_1mac, const float* sqrt_recip_alphas, const float* post_var,
                      float* out, int samples, int64_t per_sample, void* stream);
int mri_step_advance(int64_t* t, int64_t* t_prev, int n, int64_t delta, uint64_t* rng,
                     uint64_t rng_increment, void* stream);

/* ------------------------------------------------------------------------------------------
 * Backward pass (training): what autograd computes for the modules above.
 *
 * Data gradients of every convolution re-use mri_gemm_launch with transposed/flipped packed
 * weights (the adjoint of a stride-2 convolution is the parity-decomposed transposed
 * convolution and vice versa).  Weight gradients run on mri_wgrad_launch:
 *     dW[class][co][b_k + c] += sum over output positions m of dY[m, co] * A_kb[m, c]
 * for every k-table entry kb of the FORWARD plan (same a_maps, ktable, tiles, box).  dW is an
 * fp32 matrix in the packed-weight layout ([n_class][dw_rows][dw_ld]), accumulated with
 * red.global.add -- zero it first.  dy_maps: CUtensorMap[n_class], rank 5, bf16, box
 * {64, box[0..3]}, 128B swizzle (the output-gradient tensor through the forward output view).
 * ------------------------------------------------------------------------------------------ */
typedef struct MriWgradArgs {
  const void* a_maps;
  const void* dy_maps;
  const int32_t* ktable;  /* [n_class][n_kb][8], as in MriGemmArgs */
  int32_t n_kb;
  int32_t n_class;
  int32_t tiles[4];
  int32_t box[4];
  int32_t n_total;        /* valid output channels (rows of dW) */
  int32_t co_blocks;      /* ceil(n_total / 128) */
  int32_t splits;         /* CTAs sharing one dW tile (strided split of the M tiles) */
  int32_t group;          /* k-table entries per CTA, 1..4 */
  float* dw;
  int32_t dw_rows;
  int32_t dw_ld;
  int32_t stages;         /* 2..6 */
  int32_t xgroup;         /* 1: the k-table consists of kw triples (xreuse forward plans, boxes of 8 x 16
                             positions, one class); a_maps are the 10-wide maps; group = 3 or 6: each triple
                             reads ONE activation tile through an MN-major operand whose three 64-channel
                             blocks are one row apart (see gemm_wgrad.cu) */
} MriWgradArgs;
int mri_wgrad_launch(const MriWgradArgs* args_host, void* stream);

/* GroupNorm(+SiLU) backward, y = act(gn(x)*gamma+beta):
 * mri_gn_bwd_reduce: sums[3][samples][C] (fp64, accumulated with fp64 atomics so that the result
 *   does not depend on arrival order -- zero first):
 *   [0] = sum_s dy, [1] = sum_s du, [2] = sum_s du*xhat  (du = dy*act'(u)); x == NULL: only [0]
 *   (plain per-(sample, channel) column sum: bias and time-embedding-projection gradients).
 *   dgamma = sum_n sums[2], dbeta = sum_n sums[1].
 * mri_gn_bwd_apply: dx = rstd*(gamma*du - mean_g(gamma*du) - xhat*mean_g(gamma*du*xhat)) (+ add);
 *   colsum (fp64 [samples][C], may be NULL, zero it first) += sum_s dx: the bias / time-projection
 *   gradient of the convolution that produced x, for free while dx is in registers. */
int mri_gn_bwd_reduce(const void* x, const void* dy, const double* stats, const float* gamma,
                      const float* beta, double* sums, int samples, int64_t spatial, int C,
                      int groups, int stats_ld, int stats_cpg, float eps, int silu, void* stream);
int mri_gn_bwd_apply(const void* x, const void* dy, const void* add, void* dx, const double* stats,
                     const float* gamma, const float* beta, const double* sums, int samples,
                     int64_t spatial, int C, int groups, int stats_ld, int stats_cpg, float eps,
                     int silu, double* colsum, void* stream);
/* "Split" precision mode: parity with the reference's fp32 / TF32 sampling path
 * (ddpm_3d_ldm/show_model.py:254 runs the UNet without autocast).  An fp32 value travels as two
 * bf16 numbers hi = bf16(v), lo = bf16(v - hi); an activation with C channels is stored
 * channels-last as [hi | lo | hi] (3C channels) against weights [w_hi | w_hi | w_lo], so the
 * implicit-GEMM kernel (fp32 accumulation, out_f32) evaluates a_hi*w_hi + a_lo*w_hi + a_hi*w_lo.
 * mri_gn_split: v = act(GroupNorm(x)) (+ rowbias[sample, c]) (+ residual, fp32 [.., C]) of x fp32
 *   [samples, spatial, C]; stats == NULL: v = x (+ ...).  Written widened as y bf16 [samples,
 *   spatial, 3C] (y != NULL) and / or as fp32 y32 [samples, spatial, C] (y32 != NULL).  Replaces
 *   nn.GroupNorm + nn.SiLU and the adds around them (unet_attention.py:62-63,76-85;
 *   slice_cond_2d_ddpm/unet.py:44-56) in this mode; exact sigmoid.
 * mri_stats_f32: GroupNorm partial sums (sum, sum of squares; fp64 [samples][groups][2], zero it
 *   first) of an fp32 channels-last tensor whose producer is not a convolution epilogue (the 2D
 *   out_norm, slice_cond_2d_ddpm/unet.py:196).
 * mri_split3: dst[o, i, p*seg + j] = part_p(src[o, i, j]) for j < width; pattern 0 = (hi, lo, hi)
 *   (activation side), 1 = (hi, hi, lo) (weight side); leading dimensions in elements.
 * mri_softmax_rows_split: P = softmax(scale * S) per row in fp32 (unet_attention.py:49-50), written
 *   widened [hi | lo | hi] with segment length seg (ld_p >= 3 * seg).
 * mri_bf16_residual_nchw: x fp32 [B, C, S] (per_sample = C * S) -> out[b] = [x - bf16(x) | x]
 *   (2C channels; samples out_sample_stride elements apart): the extra input channels of the first
 *   convolution (unet_attention.py:114, slice_cond_2d_ddpm/unet.py:184). */
int mri_gn_split(const float* x, void* y, float* y32, const double* stats, const float* gamma,
                 const float* beta, const float* rowbias, int rowbias_ld, const float* residual,
                 int samples, int64_t spatial, int C, int groups, int stats_ld, int stats_cpg, float eps,
                 int silu, void* stream);
int mri_stats_f32(const float* x, double* stats, int samples, int64_t spatial, int C, int groups,
                  void* stream);
int mri_split3(const float* src, void* dst, int64_t outer, int inner, int width, int64_t src_outer_ld,
               int64_t src_inner_ld, int64_t dst_outer_ld, int64_t dst_inner_ld, int seg, int pattern,
               void* stream);
int mri_softmax_rows_split(const float* S, void* P, int64_t rows, int cols, int ld_s, int ld_p, int seg,
                           float scale, void* stream);
int mri_bf16_residual_nchw(const float* x, float* out, int samples, int64_t per_sample,
                           int64_t out_sample_stride, void* stream);
/* Image sizes the down-sampling factor does not divide (slice_cond_2d_ddpm/unet.py:95-99,
 * ddpm_25d_all_modalities/unet.py:95-99: `F.interpolate(x, size=skip.shape[-2:], mode="bilinear",
 * align_corners=False)` after the transposed convolution).  Channels-last bf16 [B, H, W, C], C % 8 == 0.
 * mri_copy_window_nhwc: dst[b, dh0+i, dw0+j, :] = src[b, sh0+i, sw0+j, :] (+ add at the dst index; add
 *   may alias dst) for i < nH, j < nW; the rest of dst is left alone (zero padding in front of the
 *   stride-2 convolution, cropping its output, and the adjoints of both).
 * mri_resize_bilinear_nhwc: ATen's upsample_bilinear2d with align_corners = false.
 * mri_resize_bilinear_nhwc_bwd: its adjoint, dx [B, sH, sW, C] = R^T dy [B, dH, dW, C] (+ add). */
int mri_copy_window_nhwc(const void* src, void* dst, const void* add, int B, int sH, int sW, int dH,
                         int dW, int C, int sh0, int sw0, int dh0, int dw0, int nH, int nW,
                         void* stream);
int mri_resize_bilinear_nhwc(const void* src, void* dst, int B, int sH, int sW, int dH, int dW, int C,
                             void* stream);
int mri_resize_bilinear_nhwc_bwd(const void* dy, void* dx, const void* add, int B, int sH, int sW,
                                 int dH, int dW, int C, void* stream);
/* out = a + b, bf16, n elements (multiple of 8) */
int mri_add_bf16(const void* a, const void* b, void* out, int64_t n, void* stream);
/* attention: dS = scale * P * (dP - rowsum(dP * P)); P, dS bf16 [rows][ld_p], dP fp32 [rows][ld_dp] */
int mri_softmax_bwd(const void* P, const float* dP, void* dS, int64_t rows, int cols, int ld_p,
                    int ld_dp, float scale, void* stream);
/* nn.Linear backward (fp32): dX = dZ W (if dX), dW = dZ^T X and db = sum_b dZ (if dW; overwrite) */
int mri_linear_bwd(const float* dZ, const float* X, const float* W, float* dX, float* dW, float* db,
                   int batch, int in_f, int out_f, void* stream);
int mri_silu(const float* z, float* y, int64_t n, void* stream);
int mri_silu_bwd(const float* z, const float* dy, float* dz, int64_t n, void* stream);
/* d pred of mri_minsnr_loss, scaled by the upstream gradient upstream[0] (device scalar) */
int mri_minsnr_loss_bwd(const float* pred, const float* noise, const int64_t* t, const float* snr,
                        float gamma, const float* upstream, float* dpred, int samples,
                        int64_t per_sample, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer step (torch.optim.Adam as used by ddpm_3d_ldm/train.py:243,399 and
 * slice_cond_2d_ddpm/model.py:126,167): one launch updates every parameter (fp32 p, g, exp_avg m,
 * exp_avg_sq v).  step_dev: device float holding the number of updates applied so far; the kernel
 * uses step + 1 for the bias corrections and advances it.  grad_scale / found_inf (device
 * scalars, may be NULL) implement torch.amp.GradScaler's fused protocol: g /= grad_scale, and
 * the whole update (and the step counter) is skipped when *found_inf != 0.
 * block0 = index of the segment's first 1024-element block; segs_dev lives in device memory.
 * ------------------------------------------------------------------------------------------ */
typedef struct MriAdamSeg {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
  int64_t block0;
} MriAdamSeg;
int mri_adam_step(const MriAdamSeg* segs_dev, int n_segs, int64_t total_blocks, float lr, float beta1,
                  float beta2, float eps, float weight_decay, float* step_dev, const float* grad_scale,
                  const float* found_inf, void* stream);

/* ------------------------------------------------------------------------------------------
 * Exponential moving average of the weights (optim.EMA; what DDPM / improved-diffusion /
 * diffusers' training scripts sample from): one launch updates every shadow tensor,
 * e <- lerp(e, p, w) with ATen's lerp (both of its branches, fp32, the same FMA contraction), so
 * the result equals torch._foreach_lerp_(e, p, 1 - d) -- torch.optim.swa_utils'
 * get_ema_multi_avg_fn(d) -- bit for bit.
 * count_dev: device int64 holding the number of updates applied so far; update k = count + 1
 * uses  d = decay                                           (warmup == 0)
 *       d = 0 for k = 1, min(decay, k / (9 + k)) for k >= 2 (warmup != 0; diffusers' EMAModel
 *                                                            with update_after_step = 0)
 * computed in fp64, and w = (float)(1 - d), as torch converts the Python scalar 1 - decay.  decay
 * is a double for that reason: a float 0.9999 would move w by 1.7e-4 relative.  The kernel
 * advances the counter.  found_inf (device scalar, may be NULL): when *found_inf != 0 nothing is
 * written and the counter stays -- the GradScaler skip rule of mri_adam_step.
 * block0 = index of the segment's first 1024-element block; segs_dev lives in device memory.
 * ------------------------------------------------------------------------------------------ */
typedef struct MriEmaSeg {
  float* e;
  const float* p;
  int64_t n;
  int64_t block0;
} MriEmaSeg;
int mri_ema_update(const MriEmaSeg* segs_dev, int n_segs, int64_t total_blocks, double decay,
                   int warmup, int64_t* count_dev, const float* found_inf, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Parameter-gradient finalisation: ONE launch per backward segment turns the raw products of the
 * backward kernels into `.grad` tensors in the reference layouts (what autograd leaves in
 * `param.grad` for nn.ConvNd / nn.ConvTransposeNd / nn.GroupNorm, e.g.
 * ddpm_3d_ldm/unet_attention.py:62-74).  Two segment kinds:
 *   idx != NULL: dst[i] = ((const float*)src)[idx[i]] (0 where idx[i] < 0) -- the wgrad matrix
 *                [class][Cout][source, tap, channel] re-ordered to [Cout][Cin][taps] /
 *                [Cin][Cout][taps];
 *   idx == NULL: dst[i] = (float) sum_{b < batch} ((const double*)src)[b * ld + i] -- bias and
 *                GroupNorm gamma / beta gradients from the per-(sample, channel) fp64 sums.
 * block0 = index of the segment's first 2048-element block; segs_dev lives in device memory.
 * ------------------------------------------------------------------------------------------ */
typedef struct MriFinalSeg {
  float* dst;
  const void* src;
  const int32_t* idx;
  int64_t n;
  int64_t block0;
  int32_t batch;
  int32_t ld;
} MriFinalSeg;
int mri_grad_finalize(const MriFinalSeg* segs_dev, int n_segs, int64_t total_blocks, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The data path in front of the UNets (the reference's Dataset.__getitem__ arithmetic, batched on
 * the device; reading NIfTI files stays with the host).
 *
 * mri_masked_stats: per item, over its NON-ZERO elements, mean and (population) standard deviation
 * as fp32 (two passes with fp64 sums, like numpy's) -- `mask = x != 0; mean = x[mask].mean();
 * std = x[mask].std()`
 * (slice_cond_2d_ddpm/dataset.py:71-76, ddpm_25d_all_modalities/dataset.py:84-88,
 * ddpm_3d_ldm/dataset.py:18-24).  Item i is the rows x cols view at x + i * item_stride with
 * element strides (row_stride, col_stride); either col_stride == 1 (contiguous slices / a whole
 * volume as one row) or item_stride == 1 (the slices vol[:, :, z] of an (H, W, D) NIfTI array).
 * std is replaced by 1 when it is not positive or below eps (eps = 0: the 2-D rule `std if std > 0
 * else 1.0`; eps = 1e-6: the 3-D rule `if std < eps: std = 1.0`).  An item without non-zero
 * elements gets (0, 1).  acc: fp64 scratch [items][3] (count, sum, sum of squared deviations; zeroed by the
 * call); mean_std: fp32 [items][2].
 *
 * mri_slice_normalize_resize: out[i] = 2 * bilinear(clip01(x_i)) - 1 with
 * clip01(v) = (clip(v != 0 ? (v - mean_i) / std_i : v, -5, 5) + 5) / 10 and torch's
 * F.interpolate(size=(out_h, out_w), mode="bilinear", align_corners=False)
 * (slice_cond_2d_ddpm/dataset.py:78-96, ddpm_25d_all_modalities/dataset.py:91-103).  out item i
 * is the contiguous [out_h][out_w] block at out + i * out_item_stride (so that centre and context
 * slices land directly in the channels of a [B, C, S, S] batch).
 *
 * mri_volume_normalize_patch: one modality of BraTS3DVolumeDataset._load_volume
 * (ddpm_3d_ldm/dataset.py:11-41 _normalize_volume, 44-77 _pad_to_min_shape, 80-105
 * _random_or_center_crop, 160-185) in one pass: out[z][y][x] = n(vol[z + off_d, y + off_h,
 * x + off_w]) inside the volume and 0 in the zero padding, n(v) = 2 * (clip(zscore(v), -clip,
 * clip) + clip) / (2 clip) - 1.  The volume is addressed through element strides along (D, H, W),
 * so nibabel's (H, W, D) array is read in place (stride_d = 1: transposed through shared memory);
 * off_* = crop start - pad_before (negative inside the padding).
 * ------------------------------------------------------------------------------------------ */
int mri_masked_stats(const float* x, int items, int64_t item_stride, int64_t rows, int64_t cols,
                     int64_t row_stride, int64_t col_stride, float eps, double* acc,
                     float* mean_std, void* stream);
int mri_slice_normalize_resize(const float* x, int items, int64_t item_stride, int H, int W,
                               int64_t row_stride, int64_t col_stride, const float* mean_std,
                               int out_h, int out_w, float* out, int64_t out_item_stride,
                               void* stream);
int mri_volume_normalize_patch(const float* vol, int D, int H, int W, int64_t stride_d,
                               int64_t stride_h, int64_t stride_w, const float* mean_std,
                               float clip, int off_d, int off_h, int off_w, int pd, int ph, int pw,
                               float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MRI_B200_H */
