/* adp_b200.h -- C ABI of libadp_b200.so, the sm_100a (B200) kernels behind the
 * audio_diffusion_pytorch hot path:  UNetV0 forward/backward + VDiffusion + VSampler.
 *
 * The reference (archinetai/audio-diffusion-pytorch) is pure Python and has no FFI; its
 * boundary for this path is three nn.Module factories (net_t / diffusion_t / sampler_t,
 * reference models.py:25-38).  Each entry point below replaces the arithmetic of one
 * a_unet / diffusion.py building block that those modules execute; the block it replaces
 * is cited per function (reference paths are relative to /root/reference/; "a_unet" =
 * the un-vendored third-party package, behaviour per SURVEY.md appendix A).
 *
 * Conventions
 *  - plain pointers + sizes only; every pointer is a DEVICE pointer unless stated.
 *  - activations are channels-last bf16: x[b][t][c]  (the reference is [b][c][t] fp32;
 *    the stem kernels convert at the network boundary).  fp32 for statistics/conditioning.
 *  - the caller owns every buffer (incl. workspaces); no entry point allocates or
 *    synchronises, all are CUDA-graph capturable on `stream` (a cudaStream_t).
 *  - return 0 on success, non-zero on error; adp_last_error() describes the last error of
 *    the calling thread.  There is NO CPU fallback: a non-sm_100 device is an error.
 */
#ifndef ADP_B200_H_
#define ADP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* adp_stream_t; /* cudaStream_t */

/* activation codes for adp_skinny_linear */
enum { ADP_ACT_NONE = 0, ADP_ACT_GELU = 1, ADP_ACT_SILU = 2 };

int adp_version(void);
const char* adp_last_error(void);
/* 0 iff the current CUDA device is compute capability 10.x (B200). */
int adp_device_check(void);
/* Process-wide launch switches, read when a kernel is launched (or captured into a graph):
 *  key 2: 1 = adp_conv_gemm may fetch its weights before waiting for the preceding kernel (valid
 *         while no preceding kernel writes them, e.g. in an inference graph); default 0.
 *  key 6: 1 = launch with programmatic dependent launch (PDL); 0 = plain stream order; default 1.
 * Any other key is an error. */
int adp_debug_set(int key, int value);

/* ---------------------------------------------------------------------------------------
 * adp_conv_gemm: shifted-tap GEMM on tcgen05 tensor cores (TMA -> smem -> UMMA -> TMEM).
 *   out[b,t, p*n_valid + n] = epi( sum_tap sum_k  a[b, t + off(p,tap), k] * w[p*n_pad + n, tap*c_in + k] )
 * with rows outside [0,T) reading as zero (TMA out-of-bounds fill = the conv padding).
 * Replaces (a_unet): ConvBlock's Conv1d k=3 p=1 (ResnetItem), Downsample Conv1d k=s=f (as a
 * 1-tap GEMM over the [B,T/f,f*C] view), nn.Upsample(nearest,f)+Conv1d k=3 (up_factor=f:
 * per output phase p the 3 taps collapse to <=2 taps on the low-res input, weights
 * pre-summed by the caller), every nn.Linear of Attention (to_q/to_kv/to_out), and the
 * 1x1 convs.  Epilogue: + bias[n]; * gate[b,n] (MergeModulate scale); + residual (ResnetBlock
 * shortcut / attention skip / U-Net skip); optional per-(b,group) sum & sum-of-squares of the
 * result (the next GroupNorm's statistics) accumulated into `stats`.
 */
typedef struct adp_conv_gemm_args {
  const void* a;        /* bf16 [B][T][lda]                       */
  const void* w;        /* bf16 [phases*n_pad][k_total], k_total = max_taps*c_in */
  void* out;            /* bf16 [B][T][ldo]                       */
  const float* bias;    /* fp32 [n_valid] or NULL                  */
  const void* residual; /* bf16 [B][T][ldo] or NULL               */
  const float* gate;    /* fp32 [B][ld_gate] (first n_valid used) or NULL */
  double* stats;        /* fp64 [B][groups][2] (sum, sumsq) accumulated, or NULL */
  int32_t B, T;
  int32_t c_in;         /* K per tap; multiple of 16               */
  int32_t lda, ldo;     /* row pitches in elements (multiples of 8) */
  int32_t k_total;      /* row pitch of w in elements              */
  int32_t n_pad;        /* padded outputs per phase (multiple of the N tile) */
  int32_t n_valid;      /* real outputs per phase (multiple of 8)  */
  int32_t phases;       /* 1, or up_factor                         */
  int32_t ntaps;        /* taps when up_factor <= 1 (1..3)         */
  int32_t tap_off[3];   /* row offset of each tap                  */
  int32_t up_factor;    /* 0/1: plain; f>=2: nearest-upsample-by-f + conv3 phase decomposition */
  int32_t groups;       /* GroupNorm groups for `stats` (n_valid % groups == 0) */
  int32_t block_n;      /* N tile override (16..256), 0 = auto      */
  int32_t out_fp32;     /* 1: `out` is fp32 [B][T][ldo] (conditioning projections); no residual */
  int32_t ld_gate;      /* row pitch of gate in elements (multiple of 4); 0 = n_valid */
} adp_conv_gemm_args;
int adp_conv_gemm(const adp_conv_gemm_args* args, adp_stream_t stream);

/* y = SiLU(GroupNorm(x)) -- a_unet ConvBlock's nn.GroupNorm(groups, C, eps) + nn.SiLU.
 * stats: fp64 [B][groups][2] = (sum, sumsq) over the group's channels and all T. */
int adp_gn_silu(const void* x, void* y, const double* stats, const float* gamma,
                const float* beta, int32_t B, int32_t T, int32_t C, int32_t groups, float eps,
                adp_stream_t stream);

/* Per-(b,group) sum / sumsq of a channels-last bf16 tensor, accumulated into stats. */
int adp_gn_stats(const void* x, double* stats, int32_t B, int32_t T, int32_t C, int32_t groups,
                 adp_stream_t stream);

/* y = LayerNorm_C(x; no affine, eps) * (1 + scale[b,c]) + shift[b,c]
 * -- a_unet Modulation (ModulationItem); scale_shift fp32 [B][ss_stride] with scale at
 * [0,C) and shift at [C,2C), or NULL for a plain LayerNorm (attention pre-norm; its affine
 * is folded into the following projection by the caller).  stats_out as in adp_conv_gemm. */
int adp_ln_film(const void* x, void* y, const float* scale_shift, int32_t ss_stride,
                double* stats_out, int32_t B, int32_t T, int32_t C, int32_t groups, float eps,
                adp_stream_t stream);

/* adp_ln_film plus, in the same pass, y2 = LayerNorm_C(y; no affine, eps2) of the stored y:
 * a ModulationItem followed by an AttentionItem (a_unet apex.py block order) needs both the
 * modulated tensor (the attention's residual) and its pre-norm (input of the q/k/v projection).
 * y2 == NULL degenerates to adp_ln_film. */
int adp_ln_film_dual(const void* x, void* y, void* y2, const float* scale_shift,
                     int32_t ss_stride, double* stats_out, int32_t B, int32_t T, int32_t C,
                     int32_t groups, float eps, float eps2, adp_stream_t stream);

/* o = softmax(q k^T * scale) v per (batch, head), head dim 64 -- a_unet AttentionBase.
 * q: bf16 [B][Tq][ldq] (head h at columns [h*64,(h+1)*64)), k/v likewise over Tk rows,
 * o: bf16 [B][Tq][ldo].  tcgen05 flash attention (S and O accumulators in TMEM).
 * lse: optional fp32 [B][H][Tq] = log sum_k exp(scale * q.k) per row (kept by the training
 * forward for adp_attention_bwd), or NULL. */
int adp_attention(const void* q, const void* k, const void* v, void* o, int32_t B, int32_t H,
                  int32_t Tq, int32_t Tk, int32_t ldq, int32_t ldk, int32_t ldv, int32_t ldo,
                  float scale, float* lse, adp_stream_t stream);

/* y[b][n] = out_act( sum_k in_act(x[b][k]) * w[n][k] + bias[n] ),  B <= 64 rows.
 * The step-conditioning linears: NumberEmbedder.to_out, TimeConditioningPlugin MLP,
 * Modulation.to_scale_shift and MergeModulate.to_scale of every item (a_unet).
 * x fp32 [B][ldx], w bf16 [N][ldw], y fp32 [B][ldy]. */
int adp_skinny_linear(const float* x, const void* w, const float* bias, float* y, int32_t B,
                      int32_t K, int32_t N, int32_t ldx, int32_t ldw, int32_t ldy,
                      int32_t in_act, int32_t out_act, adp_stream_t stream);

/* NumberEmbedder features: out[b] = [sigma_b, sin(2 pi sigma_b w_j), cos(2 pi sigma_b w_j), 0-pad]
 * (a_unet NumberEmbedder.forward).  out fp32 [B][ld_out], ld_out >= 2*nfreq+1. */
int adp_time_features(const float* sigma, const float* freqs, float* out, int32_t B,
                      int32_t nfreq, int32_t ld_out, adp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Network boundary ("stem") kernels: fp32 [B][C][T] <-> bf16 channels-last.
 *
 * adp_stem_in: level-0 DownsampleItem Conv1d(cx+ca -> c0, k=s=f) on cat([x, append],1)
 * (reference components.py:175 AppendChannelsPlugin + a_unet Downsample), optionally on the
 * VDiffusion-noised input x_noisy = alpha_b*x + beta_b*noise (reference diffusion.py:91).
 * Emits the GroupNorm statistics of its output. */
typedef struct adp_stem_in_args {
  const float* x;       /* fp32 [B][cx][T]                          */
  const float* append;  /* fp32 [B][ca][T] or NULL                  */
  const float* noise;   /* fp32 [B][cx][T] or NULL                  */
  const float* alpha;   /* fp32 [B] (with noise)                    */
  const float* beta;    /* fp32 [B]                                 */
  const float* w;       /* fp32 [c0][cx+ca][f]  (PyTorch Conv1d layout) */
  const float* bias;    /* fp32 [c0]                                */
  void* out;            /* bf16 [B][T/f][c0]                        */
  double* stats;        /* fp64 [B][groups][2] or NULL              */
  int32_t B, T, cx, ca, c0, f, groups;
} adp_stem_in_args;
int adp_stem_in(const adp_stem_in_args* args, adp_stream_t stream);

/* adp_stem_out: level-0 UpsampleItem (nearest f + Conv1d(c0 -> co, k=3, p=1)), SkipAdapter
 * (1x1 conv on cat([x, append]) iff cx+ca != co), MergeModulate  v = skip + gate[b]*y
 * (a_unet), then optionally, fused:
 *   - classifier-free guidance  v = v_m + (v_c - v_m)*cfg_scale  (a_unet CFG plugin;
 *     h holds 2B rows: conditional then masked),
 *   - the VSampler update (reference diffusion.py:185-187) writing x_next,
 *   - the VDiffusion loss partial sums of (v - (alpha*noise - beta*x))^2 (diffusion.py:92-95)
 *     and d(loss)/dv. */
typedef struct adp_stem_out_args {
  const void* h;        /* bf16 [Bh][T/f][c0], Bh = B (or 2B with cfg) */
  const float* x;       /* fp32 [B][cx][T]   (block input, the skip) */
  const float* append;  /* fp32 [B][ca][T] or NULL                   */
  const float* w;       /* fp32 [co][c0][3]                          */
  const float* bias;    /* fp32 [co]                                 */
  const float* w_adapt; /* fp32 [co][cx+ca] or NULL (identity skip)  */
  const float* b_adapt; /* fp32 [co] or NULL                         */
  const float* gate;    /* fp32 [Bh][ld_gate] (first co used)        */
  float* v_out;         /* fp32 [B][co][T] or NULL                   */
  /* sampler fusion */
  float* x_next;        /* fp32 [B][co][T] or NULL                   */
  const float* ab;      /* fp32 [4]: alpha_i, beta_i, alpha_{i+1}, beta_{i+1} (device) */
  /* loss fusion */
  const float* noise;   /* fp32 [B][co][T] or NULL                   */
  const float* alpha;   /* fp32 [B]                                  */
  const float* beta;    /* fp32 [B]                                  */
  double* loss_sum;     /* fp64 [1] accumulated sum of squared error */
  float* dv;            /* fp32 [B][co][T] = 2*(v - v_target)/numel, or NULL */
  float cfg_scale;      /* used iff cfg != 0                         */
  int32_t cfg;
  int32_t B, T, cx, ca, c0, co, f;
  int32_t ld_gate;      /* row pitch of gate; 0 = co                 */
} adp_stem_out_args;
int adp_stem_out(const adp_stem_out_args* args, adp_stream_t stream);

/* ResnetItem ConvBlock for narrow levels (C == 8), CUDA cores, one pass:
 *   y = Conv1d_k3(SiLU(GroupNorm(x))) + bias [+ residual]
 * then optionally the following ModulationItem on the result (LayerNorm_C + FiLM),
 * and the GroupNorm statistics of what is written.  (a_unet ConvBlock / ResnetBlock /
 * Modulation; wide levels use adp_gn_silu + adp_conv_gemm + adp_ln_film.) */
typedef struct adp_narrow_conv_args {
  const void* x;            /* bf16 [B][T][C], C in {8, 32, 64}      */
  void* y;                  /* bf16 [B][T][C]                        */
  const double* stats_in;   /* fp64 [B][groups][2]                   */
  const float* gamma;       /* fp32 [C]                              */
  const float* beta;        /* fp32 [C]                              */
  const float* w;           /* fp32 [C][C][3]                        */
  const float* bias;        /* fp32 [C]                              */
  const void* residual;     /* bf16 [B][T][C] or NULL                */
  const float* scale_shift; /* fp32 [B][ss_stride] or NULL: apply LN+FiLM */
  double* stats_out;        /* fp64 [B][groups][2] or NULL           */
  int32_t ss_stride;
  int32_t B, T, C, groups;
  float gn_eps, ln_eps;
  const void* w_packed;     /* optional, C = 32 / 64 only: the same weights as bf16
                               [C][3*C] with k = tap*C + ci (saves every block the fp32 ->
                               bf16 re-layout of w); NULL = convert from w               */
} adp_narrow_conv_args;
int adp_narrow_conv(const adp_narrow_conv_args* args, adp_stream_t stream);

/* y = bf16(SiLU(x)) elementwise: the SiLU in front of every Modulation.to_scale_shift /
 * MergeModulate.to_scale linear (a_unet), applied once to the shared feature vector. */
int adp_silu_bf16(const float* x, void* y, int64_t n, adp_stream_t stream);

/* VSampler step on its own (reference diffusion.py:185-187), for nets that do not end in
 * adp_stem_out:  x_next = a1*(a0*x - b0*v) + b1*(b0*x + a0*v),  ab = [a0,b0,a1,b1]. */
int adp_sampler_step(const float* x, const float* v, const float* ab, float* x_next, int64_t n,
                     adp_stream_t stream);

/* The sampling loop's per-step inputs selected on the device (reference diffusion.py:183-187 indexes
 * sigmas[i], alphas[i], betas[i] on the host): step[0] = iterations done since the host reset it,
 * ctrl[0] = device address of the conditioning table rows fp32 [n][ss_elems], ctrl[1] = iterations
 * sharing one table row (VInpainter resamples; 0/1 = one), ctrl[2] = n (the row index is clamped).  Copies row step/ctrl[1] to ss_out and
 * ab_table[step][0..3] to ab_out, so ONE captured graph serves every step and several steps can be
 * captured back to back.  adp_step_advance: step[0] += 1 (last launch of a step). */
int adp_step_select(const int32_t* step, const int64_t* ctrl, const float* ab_table, float* ab_out,
                    float* ss_out, int64_t ss_elems, adp_stream_t stream);
int adp_step_advance(int32_t* step, adp_stream_t stream);

/* VInpainter blend (reference diffusion.py:346-350): where mask != 0,
 * x = ab[2]*source + ab[3]*noise  (the known region re-noised to the level the sampler step just
 * produced; ab as in adp_stem_out / adp_sampler_step); elsewhere x is left as the sampler wrote it.
 * x, source, noise fp32 [n]; mask uint8 [n]. */
int adp_inpaint_blend(float* x, const float* source, const float* noise, const uint8_t* mask,
                      const float* ab, int64_t n, adp_stream_t stream);

/* ARVSampler step (reference diffusion.py:231-235), per-position noise levels.  chan fp32
 * [B, C+1, T] = the net input (channels 0..C-1 = current, channel C = sigma_i); v fp32 [B, C, T]
 * = the net output; sig_next fp32 [B, T] = sigma_{i+1}.  In place: current <- alpha_{i+1} x_pred +
 * beta_{i+1} noise_pred (alpha = cos(sigma pi/2), beta = sin(sigma pi/2)), channel C <- sig_next. */
int adp_arv_step(float* chan, const float* v, const float* sig_next, int B, int C, int T,
                 adp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * fp32 VERIFICATION MODE (B200UNet.verify_fp32, csrc/verify_f32.cu): the inference program of the
 * bf16 path -- same launch sequence, packed-weight layouts, folds -- with fp32 activations and
 * weights on simple CUDA-core kernels (exact SiLU / GELU / exp), to check the program against
 * the reference at rtol 1e-3 / atol 1e-4.  Same argument meaning as the entry point each one
 * shadows; every activation / weight pointer is fp32; GroupNorm statistics are produced by
 * adp_f32_gn_stats as a separate pass (args->stats, fused GroupNorm, noising and the fused loss
 * must be unset).  ~100x slower than the tensor-core path: never used for measurement. */
int adp_f32_conv_gemm(const adp_conv_gemm_args* args, adp_stream_t stream);
int adp_f32_gn_stats(const float* x, double* stats, int B, int T, int C, int groups, adp_stream_t stream);
int adp_f32_gn_silu(const float* x, float* y, const double* stats, const float* gamma, const float* beta,
                    int B, int T, int C, int groups, float eps, adp_stream_t stream);
/* y = LN(x; eps) * (1 + scale) + shift (scale_shift may be NULL); y2 (may be NULL) = LN(y; eps2) */
int adp_f32_ln_film(const float* x, float* y, float* y2, const float* scale_shift, int ss_stride, int B,
                    int T, int C, float eps, float eps2, adp_stream_t stream);
int adp_f32_attention(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk,
                      int ldq, int ldk, int ldv, int ldo, float scale, adp_stream_t stream);
/* y[b,n] = act_out(sum_k act_in(x[b,k]) * w[n,k] + bias[n])  (shadows adp_skinny_linear) */
int adp_f32_linear(const float* x, const float* w, const float* bias, float* y, int B, int K, int N, int ldx,
                   int ldw, int ldy, int in_act, int out_act, adp_stream_t stream);
int adp_f32_silu(const float* x, float* y, int64_t n, adp_stream_t stream);
int adp_f32_stem_in(const adp_stem_in_args* args, adp_stream_t stream);   /* args->out fp32 */
int adp_f32_stem_out(const adp_stem_out_args* args, adp_stream_t stream); /* args->h fp32 */

/* ---------------------------------------------------------------------------------------
 * Conditioning front-ends of the model wrappers (fp32, once per call, outside the step loop).
 *
 * adp_resample: polyphase windowed-sinc rate change by factor_out / factor_in (reference
 * utils.py:82-117 `resample`, used by DiffusionUpsampler.reupsample / .sample, models.py:141-165).
 * x [rows, t], bank [factor_out, taps] (taps = 2*half + factor_in, the Hann-windowed sinc
 * phases), y [rows, t_out]:  y[r, i*factor_out + p] = sum_k xpad[r, i*factor_in + k] * bank[p, k],
 * xpad = x shifted by `half` with zeros outside.  adp_resample_adjoint is its transpose
 * (dx from dy), the backward of the same op. */
int adp_resample(const float* x, const float* bank, float* y, int rows, int t, int t_out,
                 int factor_in, int factor_out, int taps, int half, adp_stream_t stream);
int adp_resample_adjoint(const float* dy, const float* bank, float* dx, int rows, int t, int t_out,
                         int factor_in, int factor_out, int taps, int half, adp_stream_t stream);

/* MelSpectrogram (reference components.py:188-236): reflect padding by `pad`, frames of n_fft
 * samples every `hop` (center=False), window [n_fft], |rFFT|, mel filterbank fb [n_fft/2+1, n_mels]
 * whose column m is non-zero on bins [band[2m], band[2m+1]); apply_log: log(max(mel, 1e-5)).
 * wave [rows, t] -> mel [rows, n_mels, frames].  n_fft: a power of two in [32, 4096]. */
int adp_mel_spectrogram(const float* wave, const float* window, const float* fb, const int32_t* band,
                        float* mel, int rows, int t, int n_fft, int hop, int pad, int frames,
                        int n_mels, int apply_log, adp_stream_t stream);

/* DiffusionVocoder.to_flat (reference models.py:194-201): ConvTranspose1d(C -> 1, kernel win,
 * stride hop, padding pad, bias-free).  spec [B, C, frames], w [C, win], out [B, t_out] with
 * t_out = (frames-1)*hop - 2*pad + win.  adp_to_flat_bwd: dspec [B, C, frames] (may be NULL) and
 * dw [C, win] (may be NULL; ACCUMULATES, zeroed by the caller) from dout [B, t_out]. */
int adp_to_flat(const float* spec, const float* w, float* out, int B, int C, int frames, int win,
                int hop, int pad, int t_out, adp_stream_t stream);
int adp_to_flat_bwd(const float* spec, const float* w, const float* dout, float* dspec, float* dw,
                    int B, int C, int frames, int win, int hop, int pad, int t_out, adp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Backward (training) entry points: VDiffusion loss.backward() through UNetV0
 * (reference diffusion.py:82-95 + autograd over the a_unet blocks).  Data gradients are
 * channels-last bf16; parameter gradients accumulate in fp32 buffers zeroed by the caller.
 * The data gradient of every conv / linear is adp_conv_gemm with transposed packed weights.
 */

/* dW[n][k] += sum_{b,t} g[b][t][g_col0+n] * x[b][t+off][x_col0+k]  (tcgen05, both operands
 * consumed MN-major in place; rows outside [0,T) read as zero).  Backward of adp_conv_gemm
 * w.r.t. one tap of W. */
typedef struct adp_wgrad_args {
  const void* g;      /* bf16 [B][T][ldg] output gradient                 */
  const void* x;      /* bf16 [B][T][ldx] forward input of the GEMM       */
  float* dw;          /* fp32 [n][ldw]                                    */
  int32_t B, T;
  int32_t n, k;       /* out / in channels of this tap                    */
  int32_t ldg, ldx, ldw;
  int32_t g_cols, x_cols; /* valid columns of g / x rows (TMA extents)    */
  int32_t g_col0, x_col0, off;
  int32_t ntaps;      /* 0/1: one tap at row offset `off`; 3: the taps off, off+1, off+2 of a k=3
                         conv in one launch, tap j written to dw + j*tap_stride                 */
  int64_t tap_stride; /* floats between the dW slabs of consecutive taps (ntaps == 3)           */
} adp_wgrad_args;
int adp_wgrad(const adp_wgrad_args* args, adp_stream_t stream);

/* GroupNorm+SiLU backward, pass 1: dxh = da*silu'(z)*gamma; dgamma += sum dz*xhat;
 * dbeta += sum dz; S[b][g] += (sum dxh, sum dxh*xhat). */
int adp_gn_silu_bwd(const void* da, const void* x, const double* stats, const float* gamma,
                    const float* beta, void* dxh, float* dgamma, float* dbeta, double* S,
                    int32_t B, int32_t T, int32_t C, int32_t groups, float eps,
                    adp_stream_t stream);
/* pass 2: dx = rstd*(dxh - S1/n - xhat*S2/n) [+ dres]; optional colsum[c] += sum dx. */
int adp_gn_bwd_apply(const void* dxh, const void* x, const double* stats, const double* S,
                     const void* dres, void* dx, float* colsum, int32_t B, int32_t T, int32_t C,
                     int32_t groups, float eps, adp_stream_t stream);
/* Modulation backward: dx, dss[b][0:C] += sum_t dy*xhat, dss[b][C:2C] += sum_t dy.
 * scale_shift == NULL: backward of the affine-free attention pre-norm; dres (bf16, optional) is a
 * gradient arriving on a parallel path (the attention's residual), added to dx. */
int adp_ln_film_bwd(const void* dy, const void* x, const float* scale_shift, int32_t ss_stride,
                    void* dx, float* dss, int32_t dss_stride, float* colsum, const void* dres,
                    int32_t B, int32_t T, int32_t C, float eps, adp_stream_t stream);
/* out[c] += sum_{b,t} x[b][t][c] * (gate ? gate[b][c] : 1)   (bias gradients) */
int adp_colsum(const void* x, const float* gate, int32_t ld_gate, float* out, int32_t B, int32_t T,
               int32_t C, adp_stream_t stream);
/* MergeModulate as its own pass (training forward keeps the pre-gate conv output y):
 * out = skip + gate[b][c]*y (+ GroupNorm statistics of out). */
int adp_skip_gate(const void* y, const void* skip, const float* gate, int32_t ld_gate, void* out,
                  double* stats, int32_t B, int32_t T, int32_t C, int32_t groups,
                  adp_stream_t stream);
/* dys = gate*dout; dgate[b][c] += sum_t dout*y. */
int adp_skip_gate_bwd(const void* dout, const void* y, const float* gate, int32_t ld_gate,
                      void* dys, float* dgate, int32_t ld_dgate, int32_t B, int32_t T, int32_t C,
                      adp_stream_t stream);
/* Backward of the concatenated conditioning projection ss = cond W^T + b:
 * dw[n][k] = sum_b dss[b][n]*cond[b][k]; dbias[n] = sum_b dss[b][n]; dcond += dss W
 * (dcond may be NULL when only the parameter gradients are wanted). */
int adp_cond_bwd(const float* dss, int32_t ld_dss, const float* cond, const void* w, float* dw,
                 float* dbias, float* dcond, int32_t B, int32_t N, int32_t K, adp_stream_t stream);

/* Backward of adp_attention (torch.autograd through a_unet AttentionBase in the reference):
 * recomputes P = exp(scale*q k^T - lse) tile by tile.  dq like q, dk / dv like k / v.
 * delta: fp32 [B][H][Tq] workspace (rowsum(dO o O), written by the call). */
typedef struct adp_attention_bwd_args {
  const void* q;        /* bf16 [B][Tq][ldq], head h at columns [h*64,(h+1)*64) */
  const void* k;        /* bf16 [B][Tk][ldk] */
  const void* v;        /* bf16 [B][Tk][ldv] */
  const void* o;        /* bf16 [B][Tq][ldo]   forward output        */
  const void* d_o;      /* bf16 [B][Tq][lddo]  gradient of o         */
  const float* lse;     /* fp32 [B][H][Tq]     from adp_attention    */
  float* delta;         /* fp32 [B][H][Tq]     workspace             */
  void* dq;             /* bf16 [B][Tq][lddq] */
  void* dk;             /* bf16 [B][Tk][lddk] */
  void* dv;             /* bf16 [B][Tk][lddv] */
  int32_t B, H, Tq, Tk;
  int32_t ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  float scale;
} adp_attention_bwd_args;
int adp_attention_bwd(const adp_attention_bwd_args* args, adp_stream_t stream);

/* The attention projections run with their LayerNorm affine folded in (Wf = W diag(g),
 * bf = W b).  Unfolds the gradients: dw[N][C] = dwf*g + dbf (x) b (stored); dg[C] += colsum(dwf o W);
 * db[C] += W^T dbf.  w, dw dense fp32 [N][C]; dwf fp32 [N][ldwf]. */
int adp_ln_fold_bwd(const float* w, const float* g, const float* b, const float* dwf, int32_t ldwf,
                    const float* dbf, float* dw, float* dg, float* db, int32_t N, int32_t C,
                    adp_stream_t stream);

typedef struct adp_narrow_conv_bwd_args {
  const void* dy;           /* bf16 [B][T][C] gradient of the conv output        */
  const void* x;            /* bf16 [B][T][C] ConvBlock input (pre GroupNorm)     */
  const double* stats_in;   /* fp64 [B][groups][2] of x                           */
  const float* gamma;
  const float* beta;
  const float* w;           /* fp32 [C][C][3]                                     */
  void* dxh;                /* bf16 [B][T][C] -> adp_gn_bwd_apply                 */
  float* dgamma;
  float* dbeta;
  double* S;                /* fp64 [B][groups][2]                                */
  float* dw;                /* fp32 [C][C][3]                                     */
  float* dbias;             /* fp32 [C]                                           */
  int32_t B, T, C, groups;
  float gn_eps;
} adp_narrow_conv_bwd_args;
int adp_narrow_conv_bwd(const adp_narrow_conv_bwd_args* args, adp_stream_t stream);

typedef struct adp_stem_out_bwd_args {
  const float* dv;          /* fp32 [B][co][T]  dL/dv (adp_stem_out's `dv`)       */
  const float* gscale;      /* fp32 [1] upstream gradient of the loss, or NULL    */
  const void* h;            /* bf16 [B][T/f][c0]                                  */
  const float* x;           /* fp32 [B][cx][T]                                    */
  const float* append;
  const float* noise;
  const float* alpha;
  const float* beta;
  const float* w;           /* fp32 [co][c0][3]                                   */
  const float* bias;
  const float* w_adapt;     /* non-NULL iff the skip adapter exists               */
  const float* gate;        /* fp32 [B][ld_gate]                                  */
  void* dh;                 /* bf16 [B][T/f][c0]                                  */
  float* dw;
  float* dbias;
  float* dgate;             /* fp32 [B][ld_dgate]                                 */
  float* dw_adapt;
  float* db_adapt;
  float* dxin;              /* optional fp32 [B][cx+ca][T]: gradient w.r.t. cat([x, append]) through
                               the skip path (identity or SkipAdapter), STORED (not accumulated) */
  int32_t B, T, cx, ca, c0, co, f, ld_gate, ld_dgate;
} adp_stem_out_bwd_args;
int adp_stem_out_bwd(const adp_stem_out_bwd_args* args, adp_stream_t stream);

typedef struct adp_stem_in_bwd_args {
  const void* dout;         /* bf16 [B][T/f][c0]                                  */
  const float* x;
  const float* append;
  const float* noise;
  const float* alpha;
  const float* beta;
  float* dw;                /* fp32 [c0][cx+ca][f]                                */
  float* dbias;             /* fp32 [c0]                                          */
  const float* w;           /* fp32 [c0][cx+ca][f] (needed for dxin) or NULL      */
  float* dxin;              /* optional fp32 [B][cx+ca][T]: += gradient w.r.t. cat([x, append])
                               (the DiffusionVocoder trains `to_flat` through append_channels,
                               reference models.py:203-209); run after adp_stem_out_bwd */
  int32_t B, T, cx, ca, c0, f;
} adp_stem_in_bwd_args;
int adp_stem_in_bwd(const adp_stem_in_bwd_args* args, adp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ADP_B200_H_ */
