/*
 * its_b200.h — C-ABI of libits_b200.so, the sm_100a kernel library behind the
 * inference-time-scaling sampling path (noise candidates -> DDPM ancestral loop
 * over the UNet -> verifier score -> best candidate).
 *
 * The reference (supyuxiang/Inference-Time-Scaling-for-Diffusion-Models-beyond-
 * Scaling-Denoising-Steps) is pure Python/PyTorch and ships no FFI; every entry
 * point below cites the reference expression(s) it replaces (file:line relative
 * to the reference root).  A maintainer binds these with ctypes — see
 * INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - no torch types, no exceptions, no exit(): each function returns 0 on
 *     success or a non-zero ITS_ERR_* code, and its_last_error_string() gives the
 *     text for the calling thread;
 *   - every launch goes to `stream` (a cudaStream_t passed as void*), nothing
 *     synchronises, nothing allocates: all entry points are CUDA-graph
 *     capturable;
 *   - activations between UNet layers are NHWC bf16 ("pixel rows" of channel
 *     vectors); the sampler state x_t, eps, noise and images are NCHW fp32 exactly
 *     as the reference holds them.
 */
#ifndef ITS_B200_H_
#define ITS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ITS_OK 0
#define ITS_ERR_INVALID 1  /* bad argument / unsupported shape            */
#define ITS_ERR_CUDA 2     /* a CUDA runtime / driver call failed          */
#define ITS_ERR_NO_DEVICE 3

#define ITS_MAX_SRC 3
#define ITS_MAX_TAPS 36
#define ITS_MAX_PHASES 4

/* library identity ------------------------------------------------------- */
int its_version(void);                     /* 10000*major + 100*minor + patch */
const char* its_last_error_string(void);   /* per-thread, never NULL          */
int its_device_sm_count(int* out_host);    /* cudaDevAttrMultiProcessorCount  */
int its_set_pdl(int32_t mode);            /* programmatic dependent launch: 0 off,
                                              1 every launch, 2 small kernels, 3
                                              tap-GEMMs only (default; env ITS_PDL) */
int its_abi_sizeof(int which);             /* 0: its_conv_desc, 1: its_src_t,
                                              2: its_phase_t (binding self-check) */

/* ------------------------------------------------------------------------
 * Fused DDPM ancestral step (one launch per sampler step).
 *   eps   = eps_u ? (1+w)*eps_c - w*eps_u : eps_c          DiffusionCondition.py:83-85
 *   mean  = c1[t]*x - c2[t]*eps                             Diffusion.py:67-72
 *   x'    = mean + sigma[t]*z   (z = 0 when t == 0)         Diffusion.py:94-99
 *   NaN check OR-reduced into *nan_flag                     Diffusion.py:100
 *   clip(x', -1, 1) on the last step when clip_last != 0    Diffusion.py:102
 * coef is a device table [T][4] of fp32 {c1, c2, sigma, 0} built from the fp64
 * schedule buffers (Diffusion.py:57-65,76-77).  t is read from *t_dev (device
 * int32) so that one captured CUDA graph can be replayed for every step.
 * w is the guidance weight as the Python float the reference holds; the kernel
 * uses float(1+w) and float(w) with separately rounded mul/mul/sub, like the
 * reference's eager ops.
 * Noise: `noise` != NULL injects z = noise[t*noise_t_stride + ...] (parity mode:
 * a [T][n_img][n_per_img] fp32 stack with noise_t_stride = n_img*n_per_img, or
 * one [n_img][n_per_img] tensor with stride 0);
 * otherwise z comes from Philox4x32-10 keyed by (seed, cand_id0 + image, t,
 * element/4) and Box-Muller, so streams do not depend on the rank count.
 * x is updated in place.
 * ---------------------------------------------------------------------- */
int its_ddpm_step(float* x, const float* eps_c, const float* eps_u,
                  const float* noise, int64_t noise_t_stride, int64_t n_img,
                  int64_t n_per_img, const float* coef, const int32_t* t_dev,
                  double w,
                  uint64_t seed, int64_t cand_id0, int32_t* nan_flag,
                  int32_t clip_last, void* stream);

/* x[i] = N(0,1) from the same Philox stream family with step tag `tag`
 * (used for x_T, neighbours and path perturbations: search_algorithm.py:67,
 * 226, 315).  out = base ? base + scale*z : scale*z.  base is [n_per_img]
 * broadcast over images when base_bcast != 0, else [n_img][n_per_img].     */
int its_philox_normal(float* out, const float* base, int32_t base_bcast,
                      float scale, int64_t n_img, int64_t n_per_img,
                      uint64_t seed, int64_t cand_id0, int32_t tag,
                      void* stream);

/* *t_dev += delta (one thread); keeps the step counter on the device.       */
int its_step_advance(int32_t* t_dev, int32_t delta, void* stream);

/* ------------------------------------------------------------------------
 * its_ddpm_step with the x0 prediction of search over paths (Ma et al.): the same
 * state update as its_ddpm_step (same kernel body, same bits), and, when x0_out
 * != NULL, from the same mixed eps and the input state x_t:
 *   x0_out = clip(r1[t]*x_t - r2[t]*eps, -1, 1)            (NaN stays NaN)
 * i.e. torch.clip(sqrt(1/abar_t)*x_t - sqrt(1/abar_t - 1)*eps, -1, 1) in fp32 with
 * separately rounded mul / mul / sub.  x0_coef is a device table [T][2] of fp32
 * {sqrt(1/abar), sqrt(1/abar - 1)} formed in fp64 from abar = cumprod(1 - betas)
 * (Diffusion.py:57-60).  The candidate base is read from *cand_dev (device int64),
 * so one captured step graph serves every round and chunk of a search.
 * ---------------------------------------------------------------------- */
int its_ddpm_step_x0(float* x, float* x0_out, const float* eps_c,
                     const float* eps_u, const float* noise,
                     int64_t noise_t_stride, int64_t n_img, int64_t n_per_img,
                     const float* coef, const float* x0_coef,
                     const int32_t* t_dev, double w, uint64_t seed,
                     const int64_t* cand_dev, int32_t* nan_flag,
                     int32_t clip_last, void* stream);

/* its_ddpm_step_x0 with one guidance weight per image, for searches over the
 * weight: image i of the launch mixes (DiffusionCondition.py:85)
 *   eps = w_img[2i+1] * eps_c - w_img[2i] * eps_u
 * with separately rounded mul / mul / sub.  w_img is a device array of n_img
 * fp32 pairs {w, 1 + w} (8-byte aligned), each formed on the host from the
 * double w as its_ddpm_step_x0 forms its scalars: (float)w, (float)(1.0 + w).
 * With every pair equal, the output is its_ddpm_step_x0's bit for bit (same
 * kernel body: posterior mean, noise, x0 prediction, NaN flag, final clip).
 * eps_u and w_img are required: the entry point only serves the guided path.
 * ---------------------------------------------------------------------- */
int its_ddpm_step_x0_w(float* x, float* x0_out, const float* eps_c,
                       const float* eps_u, const float* noise,
                       int64_t noise_t_stride, int64_t n_img, int64_t n_per_img,
                       const float* coef, const float* x0_coef,
                       const int32_t* t_dev, const float* w_img, uint64_t seed,
                       const int64_t* cand_dev, int32_t* nan_flag,
                       int32_t clip_last, void* stream);

/* Children of one search-over-paths round, q(x_s' | x_s) applied to survivors:
 *   out[i] = a * x[parent[(child0 + i) / m]] + b * z[i],   i < n_child
 * torch: a * x[parents] + b * z  (fp32, separately rounded mul / mul / add).
 * x is [n_parent][n_per], parent a device int32 array of n_sel survivor indices
 * (its_topk_first's idx_out as is), m children per survivor.  z == NULL draws z
 * from Philox (seed, cand_id0 + child0 + i, tag), the stream its_philox_normal
 * gives unit cand_id0 + child0 + i; otherwise z is [n_child][n_per].  A parent
 * index outside [0, n_parent) yields a NaN child.                           */
int its_path_expand(float* out, const float* x, const int32_t* parent,
                    int32_t n_sel, int32_t m, int64_t child0, int64_t n_child,
                    int64_t n_parent, int64_t n_per, float a, float b,
                    const float* z, uint64_t seed, int64_t cand_id0,
                    int32_t tag, void* stream);

/* ------------------------------------------------------------------------
 * Sinusoidal time embedding  emb[b,2i]=sin(t*f_i), emb[b,2i+1]=cos(t*f_i)
 * (Model.py:76-88; the table form ModelCondition.py:27-34 gives the same
 * values for integer t).  t comes from t_idx[b] (int64, host-API path) or, when
 * t_idx == NULL, from *t_dev for every row.  freq is [d_model/2] fp32.
 * ---------------------------------------------------------------------- */
int its_time_embed(float* out, const int64_t* t_idx, const int32_t* t_dev,
                   const float* freq, int32_t n_rows, int32_t d_model,
                   void* stream);

/* rows of an embedding table: out[b,:] = table[idx[b],:]  (ModelCondition.py:
 * 38, 52); idx == NULL takes row *t_dev for every b.                        */
int its_embed_rows(float* out, const float* table, const int64_t* idx,
                   const int32_t* t_dev, int32_t n_rows, int32_t dim,
                   int32_t n_table_rows, void* stream);

/* Small fp32 linear  y[b,n] (+)= sum_k act(x[b,k]) * W[n,k] + bias[n]
 * (time/cond MLPs and the per-ResBlock temb_proj/cond_proj: Model.py:38-42,
 * 181-184; ModelCondition.py:36-41, 51-56, 128-135).  silu_in applies Swish to x
 * on load; silu_out applies it to y; accumulate adds into y.                */
int its_linear(float* y, const float* x, const float* W, const float* bias,
               int32_t n_rows, int32_t K, int32_t N, int32_t silu_in,
               int32_t silu_out, int32_t accumulate, void* stream);

/* ------------------------------------------------------------------------
 * GroupNorm(32 groups) [+ Swish] over the channel concatenation of up to two
 * NHWC bf16 tensors, written as one NHWC bf16 tensor of C0+C1 channels
 * (Model.py:170-173,186-190,132,257-259 and the skip concat Model.py:279-280).
 * With stats0 (and stats1 when src1 is given) the statistics are not recomputed:
 * they are reduced, in a fixed order and in double precision, from the partial
 * sums the producing tap-GEMM wrote (its_conv_desc.stats), and the launch is one
 * streaming normalise+Swish pass (its_group_norm_apply).
 * out_fp16 bit 0: store IEEE fp16 instead of bf16.  Bits 1 and 2 say that
 * source 0 / source 1 hold IEEE fp16 (the opt-in fp16 residual stream); inputs are bf16 otherwise.
 * Deterministic (no float atomics).  chunks <= 8: ONE launch, the chunks of an
 * image form a thread-block cluster and exchange partial sums through distributed
 * shared memory; chunks > 8: two launches through `partials`, scratch of
 * n_img*chunks*groups*2 floats.
 * ---------------------------------------------------------------------- */
int its_group_norm(void* out, const void* src0, int32_t C0, const void* src1,
                   int32_t C1, const float* gamma, const float* beta,
                   int32_t n_img, int32_t HW, int32_t groups, float eps,
                   int32_t silu, float* partials, int32_t chunks,
                   int32_t out_fp16, void* stream);

int its_group_norm_apply(void* out, const void* src0, int32_t C0,
                         const float* stats0, int32_t parts0, const void* src1,
                         int32_t C1, const float* stats1, int32_t parts1,
                         const float* gamma, const float* beta, int32_t n_img,
                         int32_t HW, int32_t groups, float eps, int32_t silu,
                         int32_t out_fp16, void* stream);

/* ------------------------------------------------------------------------
 * Head / tail convolutions (CUDA-core special cases, fp32 weights).
 *   head: NCHW fp32 [n_img_in,3,H,W] -> NHWC bf16 [n_img,H,W,Cout]; image b of
 *         the output reads input image b % n_img_in (CFG: the cond and uncond
 *         halves share x_t).                                  Model.py:269
 *   tail: NHWC bf16 (already GroupNorm+Swish'ed) -> NCHW fp32 [n_img,3,H,W]
 *                                                             Model.py:257-262
 * W is the reference's OIHW fp32 tensor, unchanged.
 * ---------------------------------------------------------------------- */
int its_conv_head(void* out, const float* x, const float* W, const float* bias,
                  int32_t n_img, int32_t n_img_in, int32_t H, int32_t Wd,
                  int32_t Cin, int32_t Cout, void* stream);
/* Head on the tensor cores: the 3x3xCin patch of every pixel as one 128-channel
 * bf16 pixel [x_hi | x_lo | x_hi | 0] (x_hi = bf16(x), x_lo = bf16(x - x_hi)); a
 * 1x1 its_conv_igemm against [w_hi | w_hi | w_lo | 0] then reproduces the fp32
 * convolution of Model.py:269 to ~16 mantissa bits.  out NHWC bf16
 * [n_img][H][W][128]; image b reads input image b % n_img_in.              */
int its_head_patches(void* out, const float* x, int32_t n_img, int32_t n_img_in,
                     int32_t H, int32_t Wd, int32_t Cin, void* stream);
int its_conv_tail(float* out, const void* act, const float* W,
                  const float* bias, int32_t n_img, int32_t H, int32_t Wd,
                  int32_t Cin, int32_t Cout, void* stream);

/* ------------------------------------------------------------------------
 * Implicit-GEMM convolution / batched GEMM on tcgen05 ("tap-GEMM").
 *   D[(b,y,x), n] = alpha * sum_taps sum_c A_src[b, y*s+dy, x*s+dx, c] *
 *                   Wp[n, k(tap,c)]  + bias[n] + vec[b,n] + vec2[b,n]
 *                   + res[(b,y',x'), n]
 * over GEMM rows (b,y,x) in [B,Hm,Wm]; out pixel (y',x') = (y*os+py, x*os+px).
 * Covers ResBlock 3x3 (Model.py:170-190) with the 1x1 shortcut appended as
 * extra K (Model.py:191-194,207), DownSample 3x3 s2 (Model.py:99; +5x5 s2 summed,
 * ModelCondition.py:68-73), UpSample nearest+3x3 folded into 4 sub-pixel phases
 * (Model.py:122-125), ConvTranspose2d(5,2,2,1) as 4 phases (ModelCondition.py:
 * 80), the AttnBlock 1x1 projections and its two bmm's (Model.py:147-161).
 * Packed weights Wp are bf16 [Cout][w_pitch], K ordered (phase, tap, channel).
 * impl: 0 = tcgen05/TMA kernel, 1 = CUDA-core reference kernel (same maths;
 * debug and shapes with C % 64 != 0).
 * Layers with few output tiles (4x4 / 8x8 feature maps) can split K over
 * `splits` CTAs per tile: partial fp32 accumulators go to `ws` and a second
 * launch reduces them in a fixed order and applies the epilogue (deterministic).
 * ---------------------------------------------------------------------- */
typedef struct {
  const void* ptr;       /* bf16 [B][H][W][c_pitch]                      */
  int32_t c_pitch;       /* elements per pixel                           */
  int32_t c_off;         /* first channel used                           */
  int32_t C;             /* channels used (k-blocks of 64)               */
  int32_t H, W;          /* source spatial size                          */
  int32_t stride;        /* 1 or 2: source pixel = row pixel*stride+tap  */
  int32_t bcast;         /* 1: the same image for every b (batch size 1) */
  int32_t fp16;          /* 1: this tensor AND the weight columns of its taps
                            hold IEEE fp16 instead of bf16 (both operands of
                            an MMA must share the format).  GroupNorm
                            outputs are bounded, so they and their weights
                            use fp16's 3 extra mantissa bits; raw feature
                            maps keep bf16's range                         */
} its_src_t;

typedef struct {
  int32_t ntaps;
  int32_t w_k0;          /* first K column of this phase in Wp           */
  int32_t py, px;        /* output sub-pixel offset                      */
  int8_t src[ITS_MAX_TAPS];
  int8_t dy[ITS_MAX_TAPS];
  int8_t dx[ITS_MAX_TAPS];
} its_phase_t;

typedef struct {
  its_src_t src[ITS_MAX_SRC];
  int32_t nsrc;
  its_phase_t phase[ITS_MAX_PHASES];
  int32_t nphases;
  int32_t B, Hm, Wm;     /* GEMM rows = B*Hm*Wm                          */
  const void* w;         /* bf16 [w_batch][Cout][w_pitch]                */
  int32_t w_pitch;
  int64_t w_batch_stride;/* elements; 0 = shared weights                 */
  int32_t Cout;
  void* out;             /* bf16 or fp32 [B][Hout][Wout][out_c_pitch]    */
  int32_t out_fp32;
  int32_t Hout, Wout, out_scale, out_c_pitch, out_c_off;
  const float* bias;     /* [Cout] or NULL                               */
  const float* vec;      /* [B or 1][vec_stride] or NULL                 */
  int32_t vec_stride;    /* row stride of vec; 0 = one row for all b     */
  int32_t vec_off;       /* first column of vec used                     */
  const float* vec2;     /* second per-image vector (label embedding)    */
  int32_t vec2_stride;
  int32_t vec2_off;
  const void* res;       /* bf16, out's pixel mapping, or NULL           */
  int32_t res_c_pitch, res_c_off;
  float alpha;
  int32_t bn;            /* N tile: 0 = auto, else 32/64/128/192/256     */
  int32_t out_nchw;      /* 1: out is fp32 [B][Cout][Hout][Wout] (tail)  */
  int32_t splits;        /* split-K factor (tcgen05 path); 0/1 = none    */
  float* ws;             /* split-K scratch: nphases*splits*rows*Cout    */
  int64_t ws_elems;      /* capacity of ws in floats                     */
  int32_t cluster;       /* CTAs per cluster sharing a multicast weight tile:
                            0 = auto (4/2/1), else 1, 2 or 4             */
  int64_t* dbg;          /* diagnostics: NULL, or [CTAs][64] clock stamps
                            (scripts/conv_timeline.py)                   */
  float* stats;          /* out, optional: GroupNorm partial sums of the
                            stored bf16 tensor, [B][stats_parts][Cout/4]
                            {sum, sum of squares} (persistent schedule)   */
  int32_t stats_parts;   /* its_conv_stats_parts() of this descriptor     */
  int32_t schedule;      /* 0 = auto, 1 = one tile per CTA, 2 = persistent
                            CTAs (TMEM double buffer, TMA-store epilogue) */
  int32_t out_fp16;      /* bit 0: 16-bit NHWC output in IEEE fp16 instead of bf16 (the opt-in
                            fp16 residual stream: 3 more mantissa bits, 65504 range);
                            bit 1: `res` holds IEEE fp16                               */
  /* GroupNorm (+ Swish) of the tensor this launch computes, applied in the SAME launch's epilogue
   * (Model.py:170-173,186-190,132: the GroupNorm -> Swish that opens the next convolution or the attention
   * block reads exactly the tensor this convolution produces).  Persistent schedule only, one phase,
   * out_scale 1; see its_conv_gn_sync_words() for the shapes it covers.  The statistics are the ones
   * `stats` receives (they must be requested); a tile whose image spans several tiles waits for exactly
   * those peer tiles (consecutive work items, co-resident CTAs) through the `gn_sync` counters.        */
  void* gn_out;          /* out, optional: IEEE fp16 [B][Hm][Wm][gn_c_pitch] = Swish?(GroupNorm(D))       */
  int32_t gn_c_pitch;
  const float* gn_gamma; /* [Cout] affine weight / bias of that GroupNorm                                 */
  const float* gn_beta;
  int32_t gn_groups;     /* groups over the Cout channels (32 in both nets)                               */
  float gn_eps;
  int32_t gn_silu;       /* 1: Swish after the normalisation                                              */
  int32_t gn_only;       /* 1: `out` (the raw tensor) is not stored, only gn_out (ResBlock conv1 -> block2)*/
  int32_t* gn_sync;      /* its_conv_gn_sync_words() counters, zero-initialised ONCE (they only count up:
                            every launch adds `peers` to each), or NULL when that count is 0              */
} its_conv_desc;

int its_conv_igemm(const its_conv_desc* desc_host, int32_t impl, void* stream);

/* Number of partial-sum slots per image the persistent schedule writes into
 * desc->stats for this descriptor's tiling, or 0 when the layer cannot run on
 * the persistent schedule (no statistics are produced then).               */
int its_conv_stats_parts(const its_conv_desc* desc_host);

/* Whether the epilogue of this descriptor can apply the GroupNorm of its own output (gn_out & co.), and how many
 * peer-tile counters that takes: -1 = not fusable (run its_group_norm_apply on the stored tensor instead),
 * 0 = fusable, every tile holds whole images (4x4 / 8x8 maps), n > 0 = fusable, desc->gn_sync must point to n
 * ints zero-initialised once.  desc->gn_groups, bn, splits and schedule must already be set.                  */
int its_conv_gn_sync_words(const its_conv_desc* desc_host);

/* ------------------------------------------------------------------------
 * Attention pieces (Model.py:153-158): row softmax of fp32 scores -> bf16
 * probabilities, and a whole-block CUDA-core attention for small token counts
 * (N <= 64) where a 128-row tensor-core tile would span several images.
 * qkv is NHWC bf16 [n_img][N][3C] (q|k|v), out is [n_img][N][C].
 * ---------------------------------------------------------------------- */
int its_softmax_rows(void* probs_bf16, const float* scores, int64_t n_rows,
                     int32_t n_cols, void* stream);
int its_attention_small(void* out, const void* qkv, int32_t n_img, int32_t N,
                        int32_t C, float scale, void* stream);

/* Fused attention core for N = 256 tokens (the 16x16 maps of Model.py:153-158):
 * out[b] = softmax(scale * Q[b] K[b]^T) V[b] + bias_v, with the scores in TMEM and
 * the probabilities in shared memory only.  qk is NHWC bf16 [n_img][N][2C] (q|k),
 * vT is bf16 [n_img][C][N] (V transposed, as the V projection with the weights as
 * the A operand writes it), out is [n_img][N][C].  C a multiple of 64, <= 384. */
int its_attention_fused(void* out, const void* qk, const void* vT,
                        const float* bias_v, int32_t n_img, int32_t N, int32_t C,
                        float scale, void* stream);

/* Streaming attention core for maps with more tokens than one TMEM score tile holds
 * (ModelCondition.py:108-113 on 32x32 maps: N = 1024, C = 128): same operands and
 * result as its_attention_fused, keys processed in blocks of 128 with a running
 * row maximum / row sum (fp32); scores and probabilities stay on chip.
 * N a multiple of 128, >= 256; C = 64 or 128.                                 */
int its_attention_flash(void* out, const void* qk, const void* vT,
                        const float* bias_v, int32_t n_img, int32_t N, int32_t C,
                        float scale, void* stream);

/* Attention core for small maps (N = 16, 32 or 64 tokens: 4x4 / 8x8 maps of
 * Model.py:153-158, ModelCondition.py:108-113) on the tensor cores: 128 / N
 * consecutive images share one 128-row tile, the softmax is masked to the keys of
 * the row's own image.  qkv is the fused projection tensor [n_img][N][3C] (q|k|v,
 * bf16; the V bias is NOT folded in: it is added after the product, the rows of
 * softmax(S) sum to one), out is [n_img][N][C].  C a multiple of 64, <= 512.   */
int its_attention_group(void* out, const void* qkv, const float* bias_v,
                        int32_t n_img, int32_t N, int32_t C, float scale, void* stream);

/* ------------------------------------------------------------------------
 * Verifiers and selection.
 *   its_image_stats: per image mean, unbiased variance, min and the L2-
 *     normalised 8x8 average-pooled feature vector (verifier.py:62, 218-221,
 *     226, 277-284).  images NCHW fp32; stats [n_img][4] = {mean,var,min,|pooled|};
 *     feats [n_img][C*64] or NULL.
 *   its_candidate_scores: one score per candidate of `per_cand` consecutive
 *     images.  kind 0: 1/(1+mean var) (OracleVerifier.score, verifier.py:62-63)
 *     kind 1: 2*mean std, std halved when the candidate's min < 0
 *             (AestheticPredictor.score, verifier.py:277-286)
 *     kind 2: mean off-diagonal cosine of pooled features
 *             (SelfSupervisedVerifier.score, verifier.py:236-246)
 *   its_argmax_first: first index of the maximum, NaN never wins — the strict
 *     '>' update rule of search_algorithm.py:79-81,185-187,328-330.
 * ---------------------------------------------------------------------- */
int its_image_stats(float* stats, float* feats, const float* images,
                    int32_t n_img, int32_t C, int32_t H, int32_t W,
                    void* stream);
int its_candidate_scores(float* scores, const float* stats, const float* feats,
                         int32_t n_cand, int32_t per_cand, int32_t feat_dim,
                         int32_t kind, void* stream);
int its_argmax_first(int32_t* idx_out, float* val_out, const float* scores,
                     int32_t n, void* stream);
/* The k best candidates under the same rule (score descending, first index on ties, NaN / -inf never rank):
 * idx_out[r], val_out[r] for r < k; -1 / -inf past the number of eligible scores.  The reference keeps one
 * winner (search_algorithm.py:79-81); north_star's "top-k/argmax" — used for keeping several pivots.       */
int its_topk_first(int32_t* idx_out, float* val_out, const float* scores,
                   int32_t n, int32_t k, void* stream);
/* The same selection in n_seg independent segments, one CTA each: segment s is scores[s*seg_len, (s+1)*seg_len)
 * and its k best go to idx_out[s*k + r], val_out[s*k + r].  Indices are flat (s*seg_len + local), so the
 * output can be passed unchanged as its_path_expand's parent array over the whole population; -1 / -inf past
 * a segment's eligible scores.  Generalises the reference's per-search winner (search_algorithm.py:79-81) to
 * one winner (k = 1) or k survivors per query of a batch of searches.  its_topk_first is the n_seg = 1 case.
 * Requires n_seg, seg_len, k >= 1 and n_seg * seg_len <= INT32_MAX; no allocation, no synchronisation.   */
int its_topk_first_segmented(int32_t* idx_out, float* val_out, const float* scores,
                             int32_t n_seg, int32_t seg_len, int32_t k, void* stream);
/* Systematic resampling of Feynman-Kac particles (Singhal et al. 2025, "A General Framework for Inference-time
 * Scaling and Steering of Diffusion Models"; not in the reference), one CTA per segment (query).  Segment s is
 * reward[s*seg_len, (s+1)*seg_len); for its particle i:
 *   l_i = lam * (reward_i - carried_i)   fp32, separately rounded; carried_in == NULL means carried_i = 0
 *   w_i = exp((double)l_i - m)           in double, m the largest finite l_i; w_i = 0 when reward_i or l_i is
 *                                        not finite (NaN, +-inf)
 *   C_i = w_0 + ... + w_i                in double
 *   u   = ((c0 >> 5) * 2^26 + (c1 >> 6)) * 2^-53 in [0, 1), with (c0, c1, c2, c3) = Philox4x32-10 of the counter
 *         {s, (uint32)round, tag, (uint32)(round >> 32)} under the key {(uint32)seed, (uint32)(seed >> 32)}
 *         (the generator of its_philox_normal): one uniform per (seed, segment, round)
 *   child j < seg_len takes the smallest i with C_i > (u + j) / seg_len * C_last, evaluated without a division
 *   as seg_len * C_i > (u + j) * C_last in double (a position that rounding puts at or past C_last goes to the
 *   last i with w_i > 0; the exact rule never puts one there).
 * Outputs: ancestor_out[s*seg_len + j] = s*seg_len + i (flat, as its_topk_first_segmented's indices),
 * carried_out[s*seg_len + j] = reward_i of that ancestor (the next call's carried_in), ess_out[s] =
 * (sum w)^2 / sum w^2.  A segment with no finite weight gets ancestors -1, carried NaN and ESS 0.  Sums have a
 * fixed order and no atomics: the outputs are a deterministic function of the inputs, so every rank draws the
 * same ancestors from the same gathered rewards.  Requires n_seg, seg_len >= 1, n_seg * seg_len <= INT32_MAX,
 * lam finite and >= 0; no allocation, no synchronisation.                                                      */
int its_resample_systematic(int32_t* ancestor_out, float* carried_out, float* ess_out,
                            const float* reward, const float* carried_in, float lam,
                            int32_t n_seg, int32_t seg_len, uint64_t seed, int64_t round,
                            int32_t tag, void* stream);
/* Rank ensemble of n_members (V) verifiers (the verifier ensemble of Ma et al.; not in the reference), one CTA
 * per segment (query).  scores is candidate-major [n_seg*seg_len][V] fp32, weights a device fp32 [V] array (finite
 * and > 0, checked by the caller).  In segment s, candidate i is eligible when none of its V scores is NaN or
 * -inf (+inf is an ordinary value); E is the segment's eligible set.  For eligible i and member v:
 *   r_v(i) = |{j in E : S[j][v] < S[i][v]}| + |{j in E, j != i : S[j][v] == S[i][v]}| / 2
 *            (average ranks counted from 0: scipy's rankdata(method="average") - 1 over E)
 *   out[i] = (sum_v w_v r_v(i)) / ((sum_v w_v) (|E| - 1))  in double, member order, each product and sum
 *            separately rounded, then rounded to fp32; 1.0 when |E| = 1
 * and out[i] = NaN for an ineligible i, so it never ranks in its_topk_first_segmented.  out lies in [0, 1], higher
 * is better, and depends only on the segment's own scores.  Cost O(V seg_len^2) comparisons per segment; shared
 * memory is a fixed 8 KB tile.  Requires n_members in [1, 8], n_seg, seg_len >= 1 and n_seg * seg_len <=
 * INT32_MAX; no allocation, no synchronisation, no atomics.                                                  */
int its_rank_ensemble(float* out, const float* scores, const float* weights, int32_t n_members,
                      int32_t n_seg, int32_t seg_len, void* stream);

/* ------------------------------------------------------------------------
 * Denoising verifier: the diffusion model scores a sample by how well it
 * predicts the noise added to it at S levels t_s (the eps-prediction loss of
 * Ho et al. 2020, a Monte-Carlo estimate of the denoising ELBO), and, with the
 * guided net, by the gap between its unconditional and conditional errors (the
 * diffusion model as a zero-shot classifier, Li et al. 2023; Clark & Jaini 2023).
 * Not in the reference; the specification is tests/denoising_verifier_oracle.py.
 *   its_level_inputs: out[i*S + s] = coef[s].a * x[i] + coef[s].b * eps_tab[s]
 *     (image-major, level-minor; torch `a * x + b * eps`, fp32, separately
 *     rounded mul / mul / add).  x [n_img][n_per], eps_tab [S][n_per], coef a
 *     device [S][2] fp32 table {sqrt(abar_t), sqrt(1 - abar_t)}; out is usually
 *     the UNet plan's x_in.
 *   its_denoise_scores: one fp32 score per candidate over the UNet outputs of
 *     rows (c*per_cand + b)*S + s:  D = sum (eps[row] - eps_tab[s])^2, each
 *     difference one fp32 subtraction, squares and sums in double in a fixed
 *     order (one CTA per candidate); count = per_cand * S * n_per.
 *     eps_u == NULL: -D_c / count (likelihood); else (D_u - D_c) / count with
 *     eps_u the null-label outputs of the same rows (class).  NaN propagates.
 * Both require n_img / n_cand, per_cand, S >= 1 and n_per a positive multiple
 * of 4; no allocation, no synchronisation, no atomics.                       */
int its_level_inputs(float* out, const float* x, const float* eps_tab, const float* coef,
                     int32_t n_img, int32_t n_levels, int64_t n_per, void* stream);
int its_denoise_scores(float* scores, const float* eps_c, const float* eps_u,
                       const float* eps_tab, int32_t n_cand, int32_t per_cand,
                       int32_t n_levels, int64_t n_per, void* stream);

/* ------------------------------------------------------------------------
 * fp32-grade path (precision = "fp32").  The reference computes everything in
 * fp32 (Diffusion/Diffusion.py:74-99 over Model.py / ModelCondition.py) and
 * north_star states 1e-4 on the samples for that mode: plain CUDA-core kernels
 * over NHWC fp32 tensors, one per reference operation, fp32 FMAs in a fixed
 * order, GroupNorm statistics in double.  A parity instrument and an on-device
 * cross-check of the tcgen05 path, not the throughput path.
 *   its_f32_nchw_to_nhwc: out[b][y][x][c] = in[b % n_img_in][c][y][x]
 *   its_f32_conv2d: convolution over the channel concatenation (in0 | in1) of
 *     NHWC tensors [B][Hin][Win][C0], [..][C1]; Wt = [k*k][C0+C1][CoutP] fp32
 *     (tap, input channel, output channel; CoutP = Cout rounded up to 4);
 *     + bias[n] + vec[b*vec_stride+n] + vec2[..] + res[(b,y,x),n].
 *     mode 0: nn.Conv2d(k, stride, k/2)           Model.py:99,173,190,193,262,269
 *     mode 1: nearest x2 up-sampling, then mode 0 (stride 1)     Model.py:122-125
 *     mode 2: nn.ConvTranspose2d(k, 2, k/2, 1); Wt taps from the [Cin][Cout][k][k]
 *             weight, unflipped                                ModelCondition.py:80
 *     out NHWC fp32, or NCHW when out_nchw (the 3-channel tail, Model.py:262).
 *   its_f32_group_norm: nn.GroupNorm(groups, C0+C1) (+ Swish) of (in0 | in1),
 *     out NHWC [n_img][HW][C0+C1].            Model.py:132,170-173,186-190,257-259
 *   its_f32_attention: out[b,i,:] = softmax_j(scale q_i.k_j) v_j over the fused
 *     projection tensor qkv [n_img][N][3C].                      Model.py:147-161
 * ---------------------------------------------------------------------- */
int its_f32_nchw_to_nhwc(float* out, const float* in, int32_t n_img, int32_t n_img_in,
                         int32_t C, int32_t H, int32_t W, void* stream);
int its_f32_conv2d(float* out, const float* in0, int32_t C0, const float* in1, int32_t C1,
                   const float* Wt, const float* bias, const float* vec, int32_t vec_stride,
                   const float* vec2, int32_t vec2_stride, const float* res, int32_t B,
                   int32_t Hin, int32_t Win, int32_t Cout, int32_t k, int32_t stride,
                   int32_t mode, int32_t out_nchw, void* stream);
int its_f32_group_norm(float* out, const float* in0, int32_t C0, const float* in1, int32_t C1,
                       const float* gamma, const float* beta, int32_t n_img, int32_t HW,
                       int32_t groups, float eps, int32_t silu, void* stream);
int its_f32_attention(float* out, const float* qkv, int32_t n_img, int32_t N, int32_t C,
                      float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ITS_B200_H_ */
