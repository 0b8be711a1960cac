/* libvalle_b200.so — C ABI of the B200 (sm_100a) D3PM denoising-sampler hot path.
 *
 * The reference (csulb-datascience/TTS-with-Diffusion-model) is pure Python/PyTorch and has no
 * FFI of its own; these entry points are what a binding for the hot path replaces, one per row
 * of SURVEY.md §8(a).  Each comment cites the reference code (relative to the reference root)
 * whose arithmetic the entry point takes over.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named h_*; the caller owns all memory;
 *   - nothing here allocates device memory, synchronises the device or touches the host
 *     except for building (and caching) TMA tensor maps;
 *   - every call is stream-ordered on `stream` (a cudaStream_t) and capturable in a CUDA graph;
 *   - return value 0 = ok, negative = vb200_status; text via vb200_last_error() (thread-local);
 *   - there is no CPU fallback: without an sm_100 device the launches fail with VB200_ERR_CUDA.
 *
 * Sequence layout ("packed rows"): the reference pads to (B, T_max, d) and multiplies by a mask
 * (base.py:14-35,131,193-194,440).  Here utterances are concatenated without padding:
 * M = sum_b T_b rows, T_b = T_txt+1+T_prom+1+T_resp (base.py:277-286,427-435).
 */
#ifndef VB200_H_
#define VB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* vb200_stream_t; /* cudaStream_t */

typedef enum {
  VB200_OK = 0,
  VB200_ERR_INVALID = -1,     /* bad argument (shape, alignment, null pointer) */
  VB200_ERR_CUDA = -2,        /* CUDA runtime / driver error, launch failure */
  VB200_ERR_UNSUPPORTED = -3  /* configuration outside what the kernels implement */
} vb200_status;

typedef enum { VB200_F32 = 0, VB200_BF16 = 1, VB200_F16 = 2 } vb200_dtype;

/* GEMM epilogues (SURVEY §8b): what is fused after acc = A·Wᵀ */
typedef enum {
  VB200_EPI_NONE = 0,          /* out = acc                               (to_qkv, base.py:110)        */
  VB200_EPI_BIAS = 1,          /* out = acc + bias                        (classifier, base.py:355,440) */
  VB200_EPI_BIAS_GELU = 2,     /* out = gelu_erf(acc + bias)              (ffn.block.0+1, base.py:209-211) */
  VB200_EPI_BIAS_RESIDUAL = 3  /* out = residual + acc + bias  (fp32)     (to_out / ffn.block.3 + PrenormResidual, base.py:129,193-194) */
} vb200_epilogue;

typedef enum { VB200_ABSORBING = 0, VB200_UNIFORM = 1 } vb200_transition;

typedef enum {
  VB200_NOISE_PHILOX = 0,   /* in-kernel Philox4x32-10 keyed by (seed, step, utterance id, frame, level) */
  VB200_NOISE_UNIFORMS = 1, /* caller supplies U[0,1) float32 (n_tok, K) — the reference's torch.rand, ar_discrete.py:402,480 */
  VB200_NOISE_GREEDY = 2    /* no noise: argmax of the posterior logits */
} vb200_noise;

/* per-utterance layout record, int32[8] each (host builds it once per batch) */
enum {
  VB200_U_ROW0 = 0,   /* first packed row of the utterance                   */
  VB200_U_TTXT = 1,   /* number of phone tokens                              */
  VB200_U_TPROM = 2,  /* number of prompt frames                             */
  VB200_U_TRESP = 3,  /* number of response frames                           */
  VB200_U_TXT0 = 4,   /* offset into text_ids                                */
  VB200_U_PROM0 = 5,  /* row offset into prom_ids (rows of 8 levels)         */
  VB200_U_RESP0 = 6,  /* row offset into resp_ids / first row in the packed response-row space */
  VB200_U_GID = 7,    /* global utterance id (Philox key; invariant under sharding) */
  VB200_U_STRIDE = 8
};

const char* vb200_last_error(void);
int vb200_version(void);
/* number of SMs of the current device (grid sizing), or negative status */
int vb200_device_sms(void);

/* E1-E4 + T: token ids -> residual stream rows, fp32 (M, d).
 * Replaces Embedding.forward (base.py:237-241), MultiEmbedding.forward one-hot einsum
 * (base.py:255-274), _join with `sep` (base.py:277-286), SinusodialEmbedding.add_pe
 * (base.py:80-89) and, for the D3PM glue, time_emb (ar_discrete.py:213,752).
 *   text_w (n_text, d) bf16; prom_w (8, K, d) bf16; resp_w (n_resp_levels_w, K, d) bf16;
 *   sep (d) bf16; time_w (n_time, d) bf16 or NULL; pe (>= T_max, d) fp32 table;
 *   text_ids int32; prom_ids int32 (rows, 8); resp_ids int32 (rows, resp_levels_in);
 *   utt int32 (B, 8) records; row_utt int32 (M); t_utt int32 (B) = timestep per utterance. */
int vb200_embed_gather(float* x_out, const void* text_w, const void* prom_w, const void* resp_w,
                       const void* sep, const void* time_w, const float* pe,
                       const int32_t* text_ids, const int32_t* prom_ids, const int32_t* resp_ids,
                       const int32_t* utt, const int32_t* row_utt, const int32_t* t_utt,
                       int32_t M, int32_t d, int32_t K, int32_t resp_levels_in,
                       vb200_stream_t stream);

/* 16-bit operands.  The two operands of a GEMM are both bf16 or both fp16 (`*_dtype` = VB200_BF16 |
 * VB200_F16 names the dtype of the rows AND of the weights: tcgen05 kind::f16 faults on mixed formats).
 * fp16 has 11 significand bits against 8 and is safe for the normalised rows, the FFN hidden and the
 * classifier input (conversions saturate at +-65504) but costs power; the engine uses it for the
 * classifier input by default, which brings the full model's logits from 2.2e-2 to 1.4e-2 off the fp32
 * reference (DESIGN.md §2 has the table).  qkv, the attention output, the to_out weights and the
 * embedding tables are always bf16. */

/* N1: AdaLN.forward (base.py:145-158): h = LN(x) (no affine, eps); h = c(1-k h)h;
 * y = gamma_l * h + beta_l with table (n_rows, 2d) fp32 = [exp(log gamma) | beta] (exp applied
 * once at weight-pack time).  Row l for utterance b is level_utt[b].  out (M, d) of out_dtype.
 * `table`, `level_utt` and `row_utt` are read before the kernel waits on its predecessor in the stream
 * (programmatic dependent launch): they must not be produced by the launch immediately in front of this
 * one (the engine writes levels / timesteps once per denoise step); `x` has no such restriction. */
int vb200_adaln(void* out, vb200_dtype out_dtype, const float* x, const float* table, const int32_t* level_utt,
                const int32_t* row_utt, int32_t M, int32_t d, float eps, float k, float c,
                vb200_stream_t stream);

/* N2 (norm_type == "ln"): nn.LayerNorm(d) with affine weight/bias (base.py:175-176). */
int vb200_layernorm(void* out, vb200_dtype out_dtype, const float* x, const float* weight, const float* bias,
                    int32_t M, int32_t d, float eps, vb200_stream_t stream);

/* fp32 rows -> 16-bit rows through an index (response rows for the classifier, base.py:443,491) */
int vb200_gather_rows_bf16(void* out, vb200_dtype out_dtype, const float* x, const int32_t* row_index,
                           int32_t n_rows, int32_t d, vb200_stream_t stream);

/* A1/F1/H1 linear layers (base.py:110,129,209,214,355): out = epi(A[M,K] · W[N,K]ᵀ).
 * A and W both bf16 or both fp16 (a_dtype), row-major (nn.Linear weight layout); bias fp32 (N) or NULL; residual fp32 (M,N)
 * (may alias out); out dtype per out_dtype (BIAS_RESIDUAL requires VB200_F32).
 * tcgen05 + TMEM + TMA kernel; requires K % 8 == 0, N % 8 == 0, 16-byte aligned pointers. */
int vb200_gemm_bf16(void* out, vb200_dtype out_dtype, const void* A, vb200_dtype a_dtype, const void* W,
                    const float* bias, const float* residual, int32_t M, int32_t N, int32_t K,
                    vb200_epilogue epi, vb200_stream_t stream);

/* Same contract, plain CUDA-core kernel.  Validation aid for tests / bring-up only. */
int vb200_gemm_bf16_simt(void* out, vb200_dtype out_dtype, const void* A, vb200_dtype a_dtype, const void* W,
                         const float* bias, const float* residual, int32_t M, int32_t N,
                         int32_t K, vb200_epilogue epi, vb200_stream_t stream);

/* A1 attention core (base.py:112-127), non-causal, key padding by utterance length:
 * qkv bf16 (M, 3*n_heads*64) = [q | k | v] per row as produced by to_qkv; out bf16 (M, n_heads*64).
 * cu_rows int32 (B+1) = packed row offsets.  head_dim is 64 (every size of the model factory,
 * vall_e/vall_e/__init__.py:35-57).  scale = head_dim^-0.5 (base.py:99). */
int vb200_flash_attn_varlen(void* out_bf16, const void* qkv_bf16, const int32_t* cu_rows,
                            int32_t B, int32_t max_T, int32_t M, int32_t n_heads, float scale,
                            vb200_stream_t stream);
/* Same contract, one-warp-per-query CUDA-core kernel.  Validation aid only. */
int vb200_attn_varlen_simt(void* out_bf16, const void* qkv_bf16, const int32_t* cu_rows,
                           int32_t B, int32_t max_T, int32_t M, int32_t n_heads, float scale,
                           vb200_stream_t stream);

/* D3PM per-timestep scalar table, float32 (S, VB200_TAB_STRIDE), built on the host from the
 * fp16 transition tables (ar_discrete.py:257-277) — see vall_e/vall_e/d3pm.py.  The reverse step at t
 * reads the ONE_* fields of row t and the CUM_* fields of row t-1.  A schedule table (d3pm.schedule_table,
 * for a loop that jumps from t to s < t-1) holds Q_{t|s} = Q_{s+1}...Q_t in row t's ONE_* fields and
 * Qbar_s in row t-1's CUM_* fields; it is for the reverse-step calls only, the q_sample calls take the
 * plain table. */
enum {
  VB200_TAB_ONE_KEEP = 0,   /* Q_t[a,a]   (uniform: diagonal)            schedule table, visited t: Q_{t|s}[a,a] */
  VB200_TAB_ONE_OFF = 1,    /* Q_t[a,b]   (uniform: off-diag; absorbing: 0)                        Q_{t|s}[a,b] */
  VB200_TAB_ONE_ABSORB = 2, /* Q_t[a,m]   (absorbing only)                                         Q_{t|s}[a,m] */
  VB200_TAB_ONE_BOTH = 3,   /* Q_t[m,m]   (absorbing only)                                         Q_{t|s}[m,m] */
  VB200_TAB_CUM_KEEP = 4,   /* Qbar_t[a,a]              schedule table, row t-1 of a t that jumps to s: Qbar_s[a,a] */
  VB200_TAB_CUM_OFF = 5,    /* Qbar_t[a,b]                                                          Qbar_s[a,b] */
  VB200_TAB_CUM_ABSORB = 6, /* Qbar_t[a,m]                                                          Qbar_s[a,m] */
  VB200_TAB_CUM_BOTH = 7,   /* Qbar_t[m,m]                                                          Qbar_s[m,m] */
  VB200_TAB_LOG_KEEP = 8,   /* fp16 log(fp16(Qbar_t[a,a] + eps))   (q_sample logits)   */
  VB200_TAB_LOG_OFF = 9,
  VB200_TAB_LOG_ABSORB = 10,
  VB200_TAB_LOG_BOTH = 11,
  VB200_TAB_STRIDE = 12
};

/* Q: q_sample (ar_discrete.py:467-487): x_t = argmax_j(log(Qbar_t[x0, j] + eps) + g_j) * mask,
 * g = -log(-log(clamp(u, tiny, 1))).  Bit-exact against the reference for supplied uniforms with the
 * absorbing tables; for the uniform transition see vb200_q_sample_dense below.  x0, x_out, mask int32 (n_tok); t_tok int32 (n_tok) timestep per token. */
int vb200_q_sample(int32_t* x_out, const int32_t* x0, const int32_t* t_tok, const int32_t* mask,
                   const float* uniforms, const float* table, int32_t n_tok, int32_t K,
                   int32_t S, vb200_transition tr, vb200_stream_t stream);

/* Q against the caller's own DENSE table: log_qbar_f16 = fp16 log(Qbar_t + eps), shape (S, K, K), i.e. the
 * logits ar_discrete.py:482 forms from `q_mats` (ar_discrete.py:270-275).  Row x0 of it replaces the
 * per-timestep scalars, so the result is bit-exact against whichever dense chain product the caller holds.
 * Needed for the UNIFORM transition only: its K-term fp16 sums round differently per entry depending on the
 * summation order of the GEMM that built the table (CPU BLAS here, cuBLAS in the reference's constructor),
 * so no scalar table reproduces the last bit (absorbing products have <= 2 non-zero terms and are exact). */
int vb200_q_sample_dense(int32_t* x_out, const int32_t* x0, const int32_t* t_tok, const int32_t* mask,
                         const float* uniforms, const void* log_qbar_f16, int32_t n_tok, int32_t K,
                         int32_t S, vb200_stream_t stream);

/* q_sample with in-kernel noise (training forwards, ar_discrete.py:651-653): the same categorical
 * law — weights exp(fp16 log(Qbar_t[x0, j] + eps)) — drawn in O(1) per token from one Philox
 * uniform keyed by (seed, token index, t) instead of K Gumbel variates shipped from the host. */
int vb200_q_sample_philox(int32_t* x_out, const int32_t* x0, const int32_t* t_tok, const int32_t* mask,
                          const float* table, int32_t n_tok, int32_t K, int32_t S,
                          vb200_transition tr, uint64_t seed, vb200_stream_t stream);

/* P (standalone logits-in form): q_posterior_logits + p_sample (ar_discrete.py:347-375,401-420)
 * in closed form, O(K) per token, fp32 in registers:
 *   out_j = log(f1_j + eps) + log(f2_j + eps),  f1_j = Q_t[j, x_t],
 *   f2_j = sum_i softmax(logits)_i Qbar_{t-1}[i, j]   (t-1 clamped at 0; t == 0: raw logits, no noise)
 *   x_{t-1} = argmax_j(out_j + [t != 0] g_j).
 * logits (n_rows, ld_logits) of dtype logits_dtype; token (r, l) reads columns [l*K, (l+1)*K).
 * x_t / x_out int32 (n_rows, n_levels).  row_utt int32 (n_rows) -> utterance; t_utt int32 (B).
 * utt records give the Philox key (global utterance id, frame index).  post_out (optional, may
 * be NULL) receives the fp32 posterior logits (n_rows, n_levels, K) for parity tests. */
int vb200_posterior_sample_from_logits(int32_t* x_out, float* post_out, const void* logits,
                                       vb200_dtype logits_dtype, int64_t ld_logits,
                                       const int32_t* x_t, const int32_t* row_utt,
                                       const int32_t* t_utt, const int32_t* utt,
                                       const float* table, int32_t n_rows, int32_t n_levels,
                                       int32_t K, int32_t S, vb200_transition tr,
                                       vb200_noise noise, const float* uniforms, uint64_t seed,
                                       vb200_stream_t stream);

/* P with some x0 given (generate_audio(known_list=...): continuation, span editing, level-conditional
 * sampling).  Same arguments as vb200_posterior_sample_from_logits plus `known`, int32 (n_rows, n_levels) or
 * NULL (then exactly vb200_posterior_sample_from_logits).  known = -1: the token is drawn as there.  known = k
 * in [0, K): the token's x0 is k and it draws from the ids form of q_posterior_logits (ar_discrete.py:347-375
 * with x_start_logits=False),
 *   x_s ~ q(x_s | x_t, x0 = k)  ∝  (Q_{t|s}[j, x_t] + eps) (Qbar_s[k, j] + eps),
 * from the same table entries, eps and fp16 chain products as every other token (s = t-1 with the plain
 * table).  Its logit row is not read: it may hold anything.  Philox and greedy draws are O(1) per token (at
 * most three classes, {x_t, k, m}, weigh something of their own; greedy = the arg max, lowest class wins ties);
 * with supplied uniforms the code is the Gumbel-arg max of the K posterior logits, and post_out receives those
 * logits (0 at t == 0, where the reference returns its x_start_logits argument).  At t == 0 the code is k.
 * Philox draws are keyed by (seed, frame * n_levels + level, global utterance id, t) like every other draw. */
int vb200_posterior_sample_from_logits_known(int32_t* x_out, float* post_out, const void* logits,
                                             vb200_dtype logits_dtype, int64_t ld_logits,
                                             const int32_t* x_t, const int32_t* row_utt,
                                             const int32_t* t_utt, const int32_t* utt,
                                             const float* table, int32_t n_rows, int32_t n_levels,
                                             int32_t K, int32_t S, vb200_transition tr,
                                             vb200_noise noise, const float* uniforms, uint64_t seed,
                                             const int32_t* known, vb200_stream_t stream);

/* H1 + P in one call (SURVEY.md §8a rows H1 and P; reference base.py:355,440 followed by
 * ar_discrete.py:347-375,401-420): logits = head_in (n_rows, d) x W (n_levels*K, d)^T + bias (both bf16 or both fp16) and
 * the reverse step of vb200_posterior_sample_from_logits on them.
 * Where vb200_head_fused(d, K, noise) holds this is ONE kernel: the reverse step runs as the GEMM's
 * epilogue (streaming reservoir sampling over the column tiles of a level, see
 * csrc/head_sample_tcgen05.cu) and `logits` is not touched.  Otherwise the logits go through the
 * caller's scratch `logits` (n_rows, n_levels*K) of logits_dtype and the standalone kernel.  The Philox
 * draws of the two forms differ (both are exact samples of the same posterior); greedy codes agree up
 * to the fp16 rounding of the unfused logits. */
int vb200_head_posterior_sample(int32_t* x_out, void* logits, vb200_dtype logits_dtype,
                                const void* head_in, vb200_dtype head_in_dtype, const void* W,
                                const float* bias, int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                                const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                                const int32_t* utt, const float* table, int32_t S,
                                vb200_transition tr, vb200_noise noise, const float* uniforms,
                                uint64_t seed, vb200_stream_t stream);

/* vb200_head_posterior_sample with some x0 given: `known` int32 (n_rows, n_levels) or NULL, with the semantics of
 * vb200_posterior_sample_from_logits_known.  Same fused / unfused dispatch; in the fused kernel the classifier
 * GEMM still runs in full and the epilogue takes the O(1) draw for a known token when the two halves of its row
 * merge.  The returned codes are the step's draws: a caller that wants the given codes back overwrites the known
 * positions once after its last step (Qbar_0 = Q_0 is not the identity and eps leaks mass, so the last draw can
 * differ from k). */
int vb200_head_posterior_sample_known(int32_t* x_out, void* logits, vb200_dtype logits_dtype,
                                      const void* head_in, vb200_dtype head_in_dtype, const void* W,
                                      const float* bias, int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                                      const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                                      const int32_t* utt, const float* table, int32_t S,
                                      vb200_transition tr, vb200_noise noise, const float* uniforms,
                                      uint64_t seed, const int32_t* known, vb200_stream_t stream);

/* 1 when vb200_head_posterior_sample runs as one kernel for this configuration (K % 256 == 0,
 * 256 <= K <= 4096, d % 8 == 0, noise != VB200_NOISE_UNIFORMS), else 0.  Host-only call. */
int vb200_head_fused(int32_t d, int32_t K, vb200_noise noise);

/* Training forward's loss (SURVEY.md §8f.3; reference ar_discrete.py:684-687 `F.cross_entropy` on the
 * classifier output): loss[r, l] = -log softmax(head_in[r] W_l^T + b_l)[targets[r, l]], float32
 * (n_rows, n_levels), computed as the classifier GEMM's epilogue (online log-sum-exp over the column
 * tiles of a level; no logits in HBM).  Needs K % 256 == 0. */
int vb200_head_ce_loss(float* loss, const void* head_in, vb200_dtype head_in_dtype, const void* W,
                       const float* bias,
                       const int32_t* targets, int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                       vb200_stream_t stream);

/* Scratch the caller provides for one denoiser forward over M packed rows, M_resp of them response
 * rows (the library never allocates; reference: the activations of Base.forward base.py:427-443).
 * sizes[7] receives the byte sizes, each rounded up to 256 B, in this order:
 *   x fp32 (M, d) | h 16-bit (M, d) | qkv bf16 (M, 3d) | att bf16 (M, d) | ff 16-bit (M, 4d) |
 *   head_in 16-bit (M_resp, d) | logits logits_dtype (M_resp, n_out).
 * Returns their sum, or a negative vb200_status. */
int64_t vb200_workspace_bytes(int64_t M, int64_t M_resp, int32_t d, int32_t n_out,
                              vb200_dtype logits_dtype, int64_t* sizes);

/* Hand-off to the EnCodec decoder (SURVEY.md §8f.4; reference emb/qnt.py:32-49 `decode(codes (b q t))`,
 * fed one utterance at a time through `rearrange(resps, "t q -> 1 q t")` in decode_to_file): the packed
 * int32 codes (sum_b T_resp_b, n_levels) of a whole batch -> ONE int64 tensor (B, n_levels, T_max) in the
 * decoder's layout, frames beyond an utterance's length filled with `pad`.  utt records give each
 * utterance's first response row (VB200_U_RESP0) and length (VB200_U_TRESP). */
int vb200_codes_to_bqt(int64_t* out, const int32_t* codes, const int32_t* utt, int32_t B,
                       int32_t n_levels, int32_t T_max, int64_t pad, vb200_stream_t stream);

/* reverse-loop helper (ar_discrete.py:750): t_utt[b] -= 1 for all b, on device (graph-capturable) */
int vb200_step_timesteps(int32_t* t_utt, int32_t B, int32_t delta, vb200_stream_t stream);

/* reverse-loop helper for a loop of fewer steps than timesteps: t_utt[b] = next_t[clamp(t_utt[b], 0, S-1)] for
 * all b, on device (graph-capturable: one captured step replays for every step of a schedule).  next_t int32 (S) holds each
 * visited timestep's successor (0 after the last).  Refuses null pointers and S < 1. */
int vb200_step_timesteps_to(int32_t* t_utt, int32_t B, const int32_t* next_t, int32_t S, vb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VB200_H_ */
