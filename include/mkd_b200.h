/*
 * mkd_b200.h — C-ABI of the B200-native MakeupDiffuse denoising hot path (libmkd_b200.so).
 *
 * The reference (jiean001/MakeupDiffuse) has no native layer and no FFI: its "plugin API" for this path is
 * Python duck typing (SURVEY.md §8(b)):
 *     sampler  -> model.apply_model(x_noisy, t, cond)                      diffmk/cddim.py:16,39
 *     apply_model -> control_model(x=, hint=, timesteps=, context=)        diffmk/makeup_diffuse.py:164-165
 *                 -> diffusion_model(x=, timesteps=, context=, control=..) diffmk/makeup_diffuse.py:167-168
 * and underneath that everything is a PyTorch library call.  The entry points below are what a binding for
 * that path binds instead of those library calls: one per kernel family.  Each comment names the reference
 * operation (file:line, or the upstream lllyasviel/ControlNet op reached from the cited call site) it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers owned by the caller;
 *   - activations are NHWC ("pixel-major"): element (n,h,w,c) at ((n*H+h)*W+w)*ld + c, ld >= C;
 *   - `dtype` selects the storage type of activations/weights: MKD_BF16 (production) or MKD_F32
 *     (the fp32 check mode of BASELINE.json north_star); accumulation/statistics are always fp32;
 *     biases, norm gammas/betas and DDIM latents are always fp32;
 *   - every call is asynchronous on `stream` (a cudaStream_t), allocates nothing, retains no pointer,
 *     never synchronises the device and is CUDA-graph capturable;
 *   - return value: 0 = ok, negative = error (see MKD_E_*); mkd_last_error() gives a thread-local message.
 *     There is no CPU fallback and no other backend: a wrong architecture is MKD_E_ARCH.
 */
#ifndef MKD_B200_H
#define MKD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MKD_ABI_VERSION 12

typedef void* mkd_stream_t; /* cudaStream_t */

enum { MKD_BF16 = 0, MKD_F32 = 1 };
enum { MKD_OK = 0, MKD_E_INVALID = -1, MKD_E_ALIGN = -2, MKD_E_ARCH = -3, MKD_E_CUDA = -4, MKD_E_WORKSPACE = -5 };
enum { MKD_ACT_NONE = 0, MKD_ACT_SILU = 1, MKD_ACT_GEGLU = 2 };
enum { MKD_PATH_AUTO = 0, MKD_PATH_GENERIC = 1, MKD_PATH_TCGEN05 = 2,
       /* tests / benchmarks: force one of the two tensor-core kernels (mkd_conv2d_path reports MKD_PATH_TCGEN05 for both) */
       MKD_PATH_TCGEN05_SINGLE = 3, MKD_PATH_TCGEN05_PAIR = 4 };

/* ---- probes ------------------------------------------------------------------------------------------- */
int mkd_abi_version(void);          /* == MKD_ABI_VERSION */
int mkd_compiled_arch(void);        /* 100 : built for sm_100a only */
int mkd_device_ok(int device);      /* 0 if `device` is compute capability 10.0, else MKD_E_ARCH */
const char* mkd_last_error(void);
long long mkd_launch_count(void);   /* kernels launched by this library in this process so far (bench accounting) */

/* ---- DDIM x_t -> x_{t-1} update incl. classifier-free-guidance combine -----------------------------------
 * replaces diffmk/cddim.py:39-40 (CFG combine), :56-63 (coefficients, pred_x0), :74-78 (dir_xt, noise, x_prev).
 *   e       = cfg ? eps[0:n] + cfg_scale * (eps[n:2n] - eps[0:n]) : eps[0:n]       ([uncond; cond] order)
 *   pred_x0 = (x - sqrt_one_minus_at * e) / sqrt_at
 *   x_prev  = sqrt_a_prev * pred_x0 + dir_coef * e + (sigma_t * noise) * temperature   (noise may be NULL)
 * Every product/sum is rounded separately (no FMA contraction) so the result is bit-identical to the
 * reference's op-by-op fp32 PyTorch arithmetic.  pred_x0 may be NULL. x_prev may alias x. */
int mkd_ddim_update(const float* x, const float* eps, int cfg, float cfg_scale, const float* noise,
                    float sqrt_one_minus_at, float sqrt_at, float sqrt_a_prev, float dir_coef, float sigma_t,
                    float temperature, float* x_prev, float* pred_x0, int64_t n, mkd_stream_t stream);

/* The same update with x_prev written to n_peers (1..8) destinations: x_prev_peers is a HOST array of device pointers,
 * one per rank of the box, each pointing at this rank's slice inside that rank's gather buffer (peer memory mapped over
 * NVLink, e.g. torch symmetric memory).  The last step of a batch-sharded run thereby performs the path's only
 * collective — the all-gather of the final latents (SURVEY.md 8(e)) — with its own stores; the caller follows it with
 * a rank barrier.  Values are bit-identical to mkd_ddim_update. */
int mkd_ddim_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, const float* noise,
                          float sqrt_one_minus_at, float sqrt_at, float sqrt_a_prev, float dir_coef, float sigma_t,
                          float temperature, float* const* x_prev_peers, int n_peers, float* pred_x0, int64_t n,
                          mkd_stream_t stream);

/* ---- PLMS x_t -> x_{t-1} update (ABI v11) -------------------------------------------------------------------
 * replaces upstream ldm/models/diffusion/plms.py p_sample_plms after its model call(s): get_model_output's CFG combine,
 * the pseudo-improved-Euler / Adams-Bashforth combination of the current and up to three earlier eps, and
 * get_x_prev_and_pred_x0 (the DDIM update at sigma == 0, which PLMS requires: eta must be 0).
 *   e       = cfg ? eps[0:n] + cfg_scale * (eps[n:2n] - eps[0:n]) : eps[0:n]       ([uncond; cond] order)
 *   e_store = e                                                                    (skipped when e_store is NULL)
 *   e'      = mode 0: e                                      (plain DDIM update, e.g. the first half of step 0)
 *             mode 1: (h1 + e) / 2                           (step 0: h1 = e_t, e = e_next)
 *             mode 2: (3 e - h1) / 2
 *             mode 3: (23 e - 16 h1 + 5 h2) / 12
 *             mode 4: (55 e - 59 h1 + 37 h2 - 9 h3) / 24     (h1 = o[-1] the newest earlier e_t, h3 = o[-3] the oldest)
 *   pred_x0 = (x - sqrt_one_minus_at * e') / sqrt_at
 *   x_prev  = sqrt_a_prev * pred_x0 + dir_coef * e'
 * Every product/sum is rounded separately in upstream's order (no FMA contraction); the divisions by 2, 12 and 24 are
 * products with the fp32 reciprocals, which is how torch on CUDA evaluates a tensor divided by a Python scalar, so the
 * result is bit-identical to upstream's fp32 torch arithmetic on the GPU.  h1..h3 are read only as the mode needs them.
 * Aliasing: x_prev may alias x, and e_store may alias h3 (the ring slot of the oldest eps is overwritten by the newest);
 * no other pointers may overlap.  pred_x0 may be NULL. */
int mkd_plms_update(const float* x, const float* eps, int cfg, float cfg_scale, float* e_store, int mode, const float* h1,
                    const float* h2, const float* h3, float sqrt_one_minus_at, float sqrt_at, float sqrt_a_prev,
                    float dir_coef, float* x_prev, float* pred_x0, int64_t n, mkd_stream_t stream);

/* The same update with x_prev written to n_peers (1..8) destinations, as mkd_ddim_update_peers: the last step of a
 * batch-sharded PLMS run stores its slice of the all-gathered result into every rank's gather buffer.  Values are
 * bit-identical to mkd_plms_update. */
int mkd_plms_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, float* e_store, int mode,
                          const float* h1, const float* h2, const float* h3, float sqrt_one_minus_at, float sqrt_at,
                          float sqrt_a_prev, float dir_coef, float* const* x_prev_peers, int n_peers, float* pred_x0,
                          int64_t n, mkd_stream_t stream);

/* ---- DPM-Solver++ multistep update (ABI v12) ------------------------------------------------------------------
 * replaces upstream ldm/models/diffusion/dpm_solver/dpm_solver.py after one model call (DPMSolver with predict_x0=True,
 * method 'multistep', solver_type 'dpm_solver'): model_wrapper's classifier-free combine, data_prediction_fn at the
 * evaluated time s = t_k, and multistep_dpm_solver_update from s to the next time t = t_{k+1} of order 1
 * (dpm_solver_first_update) or 2 (multistep_dpm_solver_second_update).
 *   e       = cfg ? eps[0:n] + cfg_scale * (eps[n:2n] - eps[0:n]) : eps[0:n]       ([uncond; cond] order)
 *   m       = (x - sigma_s * e) / alpha_s                                          (the data prediction m_k)
 *   m_store = m                                                                    (skipped when m_store is NULL)
 *   order 1: x_prev = sigma_ratio * x - phi * m                      (sigma_ratio = sigma_t / sigma_s, phi = alpha_t * expm1(-h))
 *   order 2: D      = inv_r0 * (m - m_prev)                          (m_prev = m_{k-1}, inv_r0 = 1 / r0)
 *            x_prev = sigma_ratio * x - phi * m - half_phi * D       (phi = alpha_t * (exp(-h) - 1), half_phi = 0.5 * phi)
 * The scalars are the caller's, evaluated with upstream's torch expressions on the device.  Every product, sum and the
 * true division are rounded separately in upstream's order (no FMA contraction), so the result is bit-identical to
 * upstream's fp32 torch arithmetic on the GPU.  m_prev is read only for order 2.
 * Aliasing: x_prev may alias x; no other pointers may overlap (m_store and m_prev are two slots of the caller's ring). */
int mkd_dpm_update(const float* x, const float* eps, int cfg, float cfg_scale, float alpha_s, float sigma_s, float* m_store,
                   int order, const float* m_prev, float sigma_ratio, float phi, float half_phi, float inv_r0, float* x_prev,
                   int64_t n, mkd_stream_t stream);

/* The same update with x_prev written to n_peers (1..8) destinations, as mkd_ddim_update_peers: the last step of a
 * batch-sharded DPM-Solver run stores its slice of the all-gathered result into every rank's gather buffer.  Values are
 * bit-identical to mkd_dpm_update. */
int mkd_dpm_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, float alpha_s, float sigma_s,
                         float* m_store, int order, const float* m_prev, float sigma_ratio, float phi, float half_phi,
                         float inv_r0, float* const* x_prev_peers, int n_peers, int64_t n, mkd_stream_t stream);

/* ---- layout / small elementwise ---------------------------------------------------------------------------
 * NCHW fp32 (the reference boundary layout, makeup_diffuse.py:152) <-> NHWC working layout. */
int mkd_nchw_to_nhwc(const float* src, void* dst, int dtype, int N, int C, int H, int W, int ld_dst,
                     mkd_stream_t stream);
int mkd_nhwc_to_nchw(const void* src, float* dst, int dtype, int N, int C, int H, int W, int ld_src,
                     mkd_stream_t stream);
/* upstream timestep_embedding(): out[b, :] = [cos(t_b f_k), sin(t_b f_k)], optionally followed by nothing. */
int mkd_timestep_embedding(const int64_t* t, void* out, int dtype, int B, int dim, float max_period,
                           mkd_stream_t stream);
/* The same embedding of fp32 timesteps (ABI v12): upstream's `t[:, None].float() * freqs` takes fractional t as they
 * are (DPM-Solver feeds the model (t_continuous - 1/N) * 1000).  For integer t below 2^24 the result is bit-identical to
 * mkd_timestep_embedding's. */
int mkd_timestep_embedding_f32(const float* t, void* out, int dtype, int B, int dim, float max_period,
                               mkd_stream_t stream);
/* y = silu(x) on n contiguous elements (ResBlock emb_layers.0, time_embed.1). */
int mkd_silu(const void* x, void* y, int dtype, int64_t n, mkd_stream_t stream);
/* GEGLU (upstream ldm.modules.attention.GEGLU): y[m, j] = x[m, j] * gelu_erf(x[m, inner + j]). */
int mkd_geglu(const void* x, void* y, int dtype, int64_t M, int inner, int ldx, int ldy, mkd_stream_t stream);
/* y[m, c] = a[m, c] + b[m, c]  (ControlNet: h = input_blocks[0](x) + guided_hint, when not fused). */
int mkd_add(const void* a, const void* b, void* y, int dtype, int64_t M, int C, int lda, int ldb, int ldy,
            mkd_stream_t stream);

/* ---- GroupNorm(32 groups) [+ SiLU], NHWC -------------------------------------------------------------------
 * replaces upstream GroupNorm32/GroupNorm + SiLU at ResBlock.in_layers/out_layers, SpatialTransformer.norm,
 * UNet.out (reached from makeup_diffuse.py:164-168).  Statistics in fp32 over (C/groups * HW) per sample.
 * x_dtype / y_dtype may differ: tensors that are not tensor-core operands (the residual trunk, ResBlock `h`) are
 * kept in fp32 by the bf16 path so that their rounding does not accumulate; norm outputs (GEMM operands) are bf16.
 * workspace: >= mkd_groupnorm_workspace_bytes(N, groups) bytes, fp32-aligned.
 * wgroups (ABI v9; 1 = none): weight groups as in mkd_conv_desc.wgroups — with wgroups == 2 the samples n >= N/2 (N even) use
 * gamma[C .. 2C) / beta[C .. 2C): the same layer of two networks on two stacked batches in one launch.  Same parameter on
 * mkd_groupnorm_apply and on mkd_layernorm (rows m >= M/2, M even). */
size_t mkd_groupnorm_workspace_bytes(int N, int groups);
int mkd_groupnorm(const void* x, void* y, int x_dtype, int y_dtype, int N, int HW, int C, int groups, int ldx,
                  int ldy, const float* gamma, const float* beta, float eps, int silu, void* workspace,
                  size_t workspace_bytes, int wgroups, mkd_stream_t stream);


/* GroupNorm as ONE streaming pass, for inputs whose producer (mkd_conv2d with `stats`) already emitted per-tile
 * column sums: stats[((n * tiles_per_sample + t) * stats_ld + c) * 2 + {0,1}], HW == 128 * tiles_per_sample.
 * Same arithmetic as mkd_groupnorm otherwise (fp32 statistics, var = E[x^2] - mean^2 clamped at 0). */
int mkd_groupnorm_apply(const void* x, void* y, int x_dtype, int y_dtype, int N, int HW, int C, int groups, int ldx,
                        int ldy, const float* gamma, const float* beta, float eps, int silu, const float* stats,
                        int stats_ld, int tiles_per_sample, int wgroups, mkd_stream_t stream);

/* ---- LayerNorm over the last dim (BasicTransformerBlock.norm1/2/3) ---------------------------------------- */
int mkd_layernorm(const void* x, void* y, int x_dtype, int y_dtype, int64_t M, int C, int ldx, int ldy,
                  const float* gamma, const float* beta, float eps, int wgroups, mkd_stream_t stream);

/* ---- row softmax y = softmax(scale * x) over the last dim (fp32 statistics) ----------------------------------------
 * The VAE decoder's mid.attn_1 (upstream AttnBlock: one 512-wide head over all pixels, reached from decode_first_stage,
 * diffmk/makeups.py:260-262) runs as  S = Q K^T (mkd_conv2d) -> mkd_softmax_rows -> P V (mkd_conv2d).  C <= 2048. */
int mkd_softmax_rows(const void* x, void* y, int x_dtype, int y_dtype, int64_t M, int C, int ldx, int ldy, float scale,
                     mkd_stream_t stream);

/* ---- convolution / GEMM family --------------------------------------------------------------------------
 * One descriptor covers every contraction of the path: ResBlock 3x3 convs, Down (stride 2) / Up (nearest x2
 * then 3x3) convs, hint-block convs, 1x1 convs, Linear layers (H=1, W=M, R=S=1) and ControlNet zero-convs:
 *
 *   acc[n,p,q,k] = sum_{r,s,c} X[n, p*stride - pad + r, q*stride - pad + s, c] * Wt[k, r, s, c]      (fp32)
 *   v            = alpha * (acc + bias[k] + emb[n, k]) + residual[n,p,q,k]
 *   Y[n,p,q,k]   = act(v)
 *
 *   The result goes to `y` (activation dtype) and/or `y32` (fp32, pixel stride ldy32); at least one is non-NULL.
 *   bias / emb / residual may be NULL.  `residual == y` (same pointer, ldr == ldy) is the fused ControlNet
 *   injection  hs[i] += scale_i * zero_conv_i(h)  of makeup_diffuse.py:166 + upstream `hs.pop() + control.pop()`.
 *   `y` / `x` may point into a wider buffer (ld > channels): that is how skip tensors are produced straight
 *   into the decoder's concat buffers (upstream torch.cat([h, hs.pop()], 1)).
 *   act == MKD_ACT_GEGLU: Wt/bias hold K = 2*Ko rows arranged in blocks of 2*geglu_block rows
 *   (geglu_block value rows, then the geglu_block matching gate rows); Y has Ko channels:
 *   Y = v_value * gelu_erf(v_gate).  alpha/emb/residual must be unused.
 *   upsample == 1: X is first nearest-neighbour upsampled x2 (H, W are the *stored* input sizes).
 *   Weights: [K][R][S][C] ("KRSC"), dtype as activations, row pitch R*S*C elements.
 *   path: MKD_PATH_AUTO picks the tcgen05/TMA kernel when dtype == bf16 and the shape qualifies
 *   (mkd_conv2d_path tells which), else the generic kernel; the other two values force a kernel (tests). */
typedef struct mkd_conv_desc {
  int dtype;
  int N, H, W, C; /* input  */
  int K, R, S;    /* filter */
  int stride, pad, upsample;
  int ldx, ldy, ldr, lde; /* element strides: input pixel, output pixel, residual pixel, emb row */
  int act, geglu_block;
  int path;
  float alpha;
  const void* x;
  const void* w;
  void* y;
  const float* bias;
  const void* emb; /* [N, lde] activations dtype */
  const void* residual;
  int residual_dtype; /* MKD_BF16 / MKD_F32: storage type of `residual` (fp32 for trunk tensors kept unrounded) */
  int ldy32;
  float* y32;         /* optional fp32 copy of the output (same values before rounding); `y` may then be NULL */
  void* workspace; /* split-K partials (tcgen05 path); may be NULL -> no split-K */
  size_t workspace_bytes;
  /* optional GroupNorm statistics of the output, fused into the tcgen05 epilogue (act must be NONE, K % 8 == 0):
   * stats[(t * stats_ld + k) * 2 + {0, 1}] = (sum, sum of squares) over rows [128 t, 128 t + 128) of the values
   * stored for output channel k.  The consumer is mkd_groupnorm_apply.  `stats` may point into a wider statistics
   * row (stats_ld > K) the same way `y` may point into a concat buffer.  Not available on the generic path. */
  float* stats;
  int stats_ld;
  /* extra zero padding on the bottom / right edge only (0 or 1).  The VAE encoder's Downsample is
   * F.pad(x, (0,1,0,1)) followed by a 3x3 stride-2 conv without padding: pad = 0, pad_hi_extra = 1. */
  int pad_hi_extra;
  /* optional second 1x1 term over another input with the output's pixels (ABI v8; NULL = absent):
   *   acc[n,p,q,k] += sum_{c < C2} X2[n,p,q,c] * Wt[k][R*S*C + c]
   * The weight rows are then [R][S][C] followed by C2 more columns (row pitch R*S*C + C2) and `bias` is the sum of the
   * two layers' biases.  This is a ResBlock's `out_layers` 3x3 conv and its 1x1 `skip_connection` (upstream
   * ldm ResBlock._forward: `self.skip_connection(x) + h`) as ONE contraction: the skip projection neither runs as its own
   * GEMM nor travels through memory as an fp32 tensor.  stride must be 1, C2 % 64 == 0, ldx2 % 8 == 0; only the tensor-core
   * CTA-pair kernel takes it: mkd_conv2d_path() returns MKD_E_INVALID when that kernel declines the shape (the caller then
   * issues the two layers separately). */
  const void* x2;
  int C2, ldx2;
  /* weight groups (ABI v9; 0 or 1 = none, 2 = two groups): the output rows are split in `wgroups` equal, contiguous parts and
   * part g is computed with weight rows [g*K, (g+1)*K) of `w` and bias[g*K .. (g+1)*K): ONE launch evaluates the same layer
   * of two networks on two stacked batches — the ControlNet trunk is a copy of the UNet encoder (cldm.ControlNet.__init__
   * mirrors UNetModel's input_blocks / middle_block), and makeup_diffuse.py:164-168 runs both on the same x_t every step.
   * `w` holds wgroups*K rows, `bias` wgroups*K values; emb / residual / y / stats are indexed by output row as always.
   * Only the tensor-core CTA-pair kernel takes it, with whole 256-row tile pairs per part: mkd_conv2d_path() returns
   * MKD_E_INVALID otherwise and the caller issues one launch per part on row / weight-row slices. */
  int wgroups;
  /* GroupNorm tail (ABI v10; gn_y == NULL: none).  Where the library runs the layer as split-K partials + reducer (the 8x8 / 4x4
   * levels at small batch), the reducer — which already reads every output value once — also normalises it: one thread block
   * per (image, group) sums the partials, applies bias / emb / alpha / residual, stores y / y32 as usual, reduces mean and
   * variance of the group in fp32 and writes
   *     gn_y[m, k] = (silu?)( (v[m, k] - mean[n, g]) * rstd[n, g] * gn_gamma[k] + gn_beta[k] )        (activation dtype)
   * i.e. the GroupNorm32(+SiLU) that follows the conv in a ResBlock (upstream ldm ResBlock.out_layers[0:2]) without its own launch
   * and without re-reading the conv output.  With wgroups == 2, gn_gamma / gn_beta hold [2, K] like mkd_groupnorm's.
   * act must be NONE, (K / gn_groups) % 8 == 0, pixels per image * K / gn_groups / 8 <= 512.  Only launches that split K carry
   * it: mkd_conv2d_path() returns MKD_E_INVALID otherwise and the caller runs mkd_groupnorm after the conv. */
  void* gn_y;
  int gn_ld, gn_groups, gn_silu;
  float gn_eps;
  const float* gn_gamma;
  const float* gn_beta;
} mkd_conv_desc;

int mkd_conv2d(const mkd_conv_desc* d, mkd_stream_t stream);
int mkd_conv2d_path(const mkd_conv_desc* d); /* MKD_PATH_GENERIC or MKD_PATH_TCGEN05, or <0 on invalid desc */

/* ---- attention (SpatialTransformer attn1 self / attn2 cross; upstream CrossAttention.forward) -------------
 *   O[b, i, h*d:(h+1)*d] = softmax_j( scale * <Q[b,i,h], K[b,j,h]> ) V[b,j,h]      softmax in fp32
 * Q rows: q + (b*Nq + i)*ldq + h*d ; K/V rows: k + (b*Nkv + j)*ldk + h*d (so q/k/v may be column slices of one
 * fused projection buffer).  d % 8 == 0, d <= 512: head dims up to 160 (the SpatialTransformer's) run on the tensor
 * cores in bf16, wider single heads (the VAE decoder's 512-wide mid.attn_1) on the one-warp-per-query SIMT kernel. */
int mkd_attention(const void* q, const void* k, const void* v, void* o, int dtype, int B, int heads, int Nq,
                  int Nkv, int d, int ldq, int ldk, int ldv, int ldo, float scale, mkd_stream_t stream);

/* ---- conditioning producer (SURVEY.md 8(f) rank 3): FrozenCLIPEmbedder (yaml:109-110; makeup_controlnet.py:20) ----
 * Runs once per prompt, not per step.  (ABI v6)
 * mkd_embed_tokens: out[b*T + t, :] = tok_emb[ids[b*T + t], :] + pos_emb[t, :]  — CLIPTextEmbeddings.forward; fp32
 *   tables and output, C % 4 == 0, ids must lie in [0, vocab).
 * mkd_attention_causal: mkd_attention with Nq == Nkv == N and key j visible to query i iff j <= i — the causal mask of
 *   CLIPTextTransformer; N short (77), one warp per query row. */
int mkd_embed_tokens(const int64_t* ids, const float* tok_emb, const float* pos_emb, float* out, int B, int T, int C,
                     int vocab, int ld_out, mkd_stream_t stream);
int mkd_attention_causal(const void* q, const void* k, const void* v, void* o, int dtype, int B, int heads, int N, int d,
                         int ldq, int ldk, int ldv, int ldo, float scale, mkd_stream_t stream);

/* ---- test-harness output (SURVEY.md 8(f) rank 4): `save_local`, diffusion_makeup.py:344-358 (ABI v6) -----------------
 * images: N x C x H x W fp32 (C = 1 or 3) -> grid: GH x GW x 3 uint8, GH = (H + padding) * ceil(N / min(nrow, N)) + padding,
 * GW = (W + padding) * min(nrow, N) + padding: torchvision make_grid (pad_value 0), optional clamp to [-1, 1], optional
 * (x + 1) / 2, x * 255 truncated to uint8 — byte-identical to the reference's torch / numpy sequence (N == 1: no padding
 * frame, as make_grid returns a single image unchanged). */
int mkd_image_grid_u8(const float* images, unsigned char* grid, int N, int C, int H, int W, int nrow, int padding, int clamp,
                      int rescale, mkd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MKD_B200_H */
