/* libwavjepa_b200.so -- C ABI of the B200-native WavJEPA hot path.
 *
 * The reference (labhamlet/wavjepa) is pure Python/PyTorch and has NO FFI layer: its boundary for this path is the
 * Python module API (wavjepa/jepa.py JEPA, wavjepa/extractors/*, wavjepa/masking.py, hear_api/runtime.py).  This
 * header is therefore the boundary a maintainer would bind from that Python (ctypes stub shown in INTEGRATION.md);
 * every entry point cites the reference op (file:line under the reference checkout) it replaces.
 *
 * Conventions: raw device pointers + explicit sizes; the caller owns every buffer; every function is asynchronous on
 * the given cudaStream_t (passed as void*), never synchronises the device, keeps no global mutable state besides
 * immutable function attributes; returns 0 on success, <0 on error with wj_last_error() giving a thread-local message.
 * There is no CPU fallback: on a machine without an sm_100 device every compute entry point fails.
 */
#ifndef WAVJEPA_B200_H
#define WAVJEPA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WJ_OK 0
#define WJ_ERR_ARG (-1)
#define WJ_ERR_RUNTIME (-2)
#define WJ_ERR_ARCH (-3)

const char* wj_last_error(void);
int wj_version(void);
/* Number of CUDA kernels this library has launched in the calling process so far (bench.py: gpu_launches). */
long long wj_kernel_launches(void);
/* 0 if the current device is sm_100 (B200); WJ_ERR_ARCH otherwise. */
int wj_check_device(void);

/* ------------------------------------------------------------------------------------------------------------------
 * GEMM operand description (bf16).  A 4-D strided view, innermost dimension first:
 *   dim[0] = contiguous "virtual column" extent of one segment, dim[1] = parity/sub-row selector, dim[2] = rows per
 *   batch entry, dim[3] = batch.  stride_bytes[i] is the byte stride of dim[i+1].
 * Virtual columns vc are split in segments of seg_width (0 = one segment); segment s addresses
 *   (vc % seg_width, seg_q[s], row + seg_p[s], batch) -- this is what turns the strided Conv1d windows of
 *   wavjepa/extractors/audio_feature_extractor.py:70 into plain TMA tiles over channels-last activations.
 * Out-of-range coordinates (including negative rows) read as zero.
 */
typedef struct wj_operand {
  const void* ptr;
  int64_t dim[4];
  int64_t stride_bytes[3];
  int32_t seg_width;
  int32_t seg_q[4];
  int32_t seg_p[4];
} wj_operand_t;

/* Fused epilogue of wj_gemm_bf16, applied in this order:
 *   v = acc + bias[n]
 *   act == 1 : h = bf16(v); out2[row, n] = bf16(GELU_erf'(h)) (if out2); v = GELU_erf(h)   (nn.GELU, types/wavjepa_configs.py:37)
 *   act == 2 : v = v * aux[row, n]            (backward of the above: aux = the GELU' saved in out2 by the forward)
 *   act == 3 : v = bf16(v)                         (autocast: the Linear output is bf16 before the fp32 residual add)
 *   v += resid[row % resid_mod or row, n]                                        (residual / positional table)
 *   out[row, n] = v  (bf16, or fp32 when out_f32; fp32 reduce-add when accumulate)
 *   colsum[n] += sum_rows out[row, n]  (optional, fp32 atomics: the bias gradient of the layer that produced `out`)
 * out_rows (optional, int32 per logical row): physical row used for out/out2/resid/aux, <0 skips the row.
 */
typedef struct wj_epilogue {
  void* out;
  int64_t ld_out;
  int32_t out_f32;
  int32_t accumulate;
  void* out2;
  int64_t ld_out2;
  const float* bias;
  const void* resid;
  int32_t resid_f32;
  int32_t resid_mod;
  int64_t ld_resid;
  const void* aux;
  int64_t ld_aux;
  int32_t act;
  int32_t _pad;
  const int32_t* out_rows;
  float* colsum;
} wj_epilogue_t;

/* out[b*L + t, n] = epilogue( sum_vc A(vc; t, b) * W[n, vc] ),  W bf16 [N, K] row-major with leading dim ldw.
 * tcgen05.mma (cta_group::1, 128 x block_n x 16) fed by TMA, fp32 accumulation in TMEM.
 * Replaces: F.linear under bf16 autocast (nn.TransformerEncoderLayer / nn.MultiheadAttention projections built at
 * wavjepa/jepa.py:126-132) and nn.Conv1d(512,512,k,stride 2) (audio_feature_extractor.py:70) as implicit GEMM. */
int wj_gemm_bf16(const wj_operand_t* A, const void* W, int64_t ldw, int L, int batch, int N, int K,
                 const wj_epilogue_t* epi, int block_n, void* stream);

/* out[b*L + t, n] = epilogue( sum_{s,r} A(s*seg_width + r; t, b) * W[r, seg_col_off[s] + n] ): the reduction runs over the
 * ROWS of the row-major bf16 matrix W [w_rows, w_cols] (read MN-major), i.e. dX = dY W for y = x W^T with no
 * transposed weight copy; with segments it is the data gradient of the stride-2 Conv1d layers. */
int wj_gemm_dgrad_bf16(const wj_operand_t* A, const void* W, int64_t ldw, int w_rows, int w_cols,
                       const int32_t* seg_col_off, int L, int batch, int N, int K, const wj_epilogue_t* epi,
                       int block_n, void* stream);

/* Deterministic mode.  By default reductions over rows / tokens / blocks end in floating-point atomics (split-token weight
 * gradients, bias column sums, LayerNorm gamma/beta gradients, the mask-token gradient, the conv-0 reduction, the loss and
 * gradient-norm scalars), so their low-order bits depend on the order in which blocks finish.  With a workspace
 * registered here (device memory, >= 256 MB covers the 512-instance training step) every such reduction stores per-block
 * or per-split partial results in the workspace and a second kernel adds them in a fixed order: two runs on the same inputs
 * give bit-identical gradients and parameters.  The workspace is used by whichever call runs, so calls must be issued on
 * ONE stream while the mode is on.  workspace = NULL (or bytes = 0) switches the mode off (the default). */
int wj_set_deterministic(void* workspace, size_t bytes);

/* Routing switches for A/B measurements and tests: key 1 = weight-gradient GEMMs may use the CTA-pair kernel, key 2 = data
 * gradient GEMMs may (value 1, the default) or stay on single CTAs (value 0). */
int wj_gemm_option(int key, int value);

/* Development aid (profiles/r02_gemm_cycle_counters.txt): `counters` = device buffer of 8 int64 per CTA that the
 * single-CTA GEMM launches after this call fill with clock64 counters of their MMA / producer / epilogue roles (time spent
 * waiting for operands, for a free accumulator, for a free stage); NULL (default) switches them off. */
int wj_gemm_debug(void* counters);

/* dW[m, vc] (+)= sum_{b,t} dY[b, t, m] * X(vc; t, b)   fp32 out [M, N] (leading dim ld_out); both operands are read
 * MN-major straight from the row-major activations; the token reduction is split over `splits` CTAs (0 = auto) and
 * reduced with red.global.add.  Replaces autograd's weight gradients of the Linear / Conv1d layers above. */
int wj_gemm_wgrad_bf16(const wj_operand_t* dY, const wj_operand_t* X, int L, int batch, int M, int N, float* out,
                       int64_t ld_out, int accumulate, int splits, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Mask generation, bit-exact with the reference maskers for the same seed (integer kernels, one warp per row).
 * kind 0 = TimeInverseBlockMasker.forward (wavjepa/masking.py:66-128), kind 1 = SpeechMasker.forward (:167-207),
 * both on top of compute_mask_indices (wavjepa/audio_masking.py:5-194) and numpy's SeedSequence/PCG64/choice chain.
 * Seed contract: call c (0 = context, 1..G = targets) of attempt a of global row r = row0 + i draws from
 * numpy.random.default_rng([base_seed, r, a*8 + c]).
 * Outputs are torch.bool-compatible bytes: ctx_hidden [batch, T_out] (True = masked context), tgt [batch, G, T_out]
 * (True = predict), vis_hidden [batch, G, T_out] (True = hidden from the predictor); T_out = n_times when
 * channel_based ("(S C)" interleave, masking.py:120-126) else n_times / in_channels.  attempts (optional) receives the
 * number of rejection-loop attempts per row; *err_flag is set to 1 if a row could not be generated. */
int wj_masks_generate(int kind, int batch, int n_times, int in_channels, int channel_based, int n_targets,
                      double ctx_prob, int ctx_len, double tgt_prob, int tgt_len, float cutoff, int min_context_len,
                      uint32_t base_seed, uint32_t row0, uint8_t* ctx_hidden, uint8_t* tgt, uint8_t* vis_hidden,
                      int* attempts, int* err_flag, void* stream);

/* Packed token index lists for the variable-length kernels (replaces the boolean gathers / scatters of
 * wavjepa/jepa.py:399 and :425-435).  For B instances, G target groups, T tokens:
 *   n_c[B], cu_c[B+1]      visible context tokens per instance;  ctx_rows[Nc] = b*T + t
 *   n_v[B*G], cu_v[B*G+1]  predictor tokens per (b, g) (visible = !vis_hidden); vis_src[Nv] = packed context index
 *                          or -1 (mask token), vis_pos[Nv] = t
 *   n_t[B*G], cu_t[B*G+1]  target tokens per (b, g); tgt_vrow[Nt] = row in the packed predictor array,
 *                          tgt_trow[Nt] = b*T + t (row of the teacher targets)
 *   totals[8] = {Nc, Nv, Nt, #targets hidden from the predictor (unsupported, must be 0), max n_c, max n_v, 0, 0} */
int wj_mask_indices(const uint8_t* ctx_hidden, const uint8_t* tgt, const uint8_t* vis_hidden, int B, int G, int T,
                    int* n_c, int* n_v, int* n_t, int* cu_c, int* cu_v, int* cu_t, int* totals, int* ctx_rows,
                    int* vis_src, int* vis_pos, int* tgt_vrow, int* tgt_trow, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Waveform encoder block 0: Conv1d(Cin->C, k=10, s=5, no bias) + GroupNorm(C, C, eps) + exact GELU, fused, output
 * channels-last bf16 [B, L_out, C].  x is [B, Cin, L] bf16, w the fp32 master weight [C, Cin, 10] (rounded to bf16 on
 * load, as autocast does).  Workspaces written by the forward and consumed by the backward:
 *   moments [B, wj_conv0_moment_count(Cin)] fp64: window sums s[a] and second moments R[a][a'] of the input
 *   stats   [B, C, 2] fp32: GroupNorm (mean, rstd) of every (instance, channel), closed form from the moments.
 * Reference: wavjepa/extractors/audio_feature_extractor.py:70,94,95. */
int wj_conv0_moment_count(int Cin);
int wj_conv0_gn_gelu_fwd(const void* x_bf16, const float* w, const float* gamma, const float* beta, int B, int Cin,
                         int L, int C, int k, int stride, float eps, double* moments, float* stats, void* out_bf16,
                         void* dgelu_bf16, void* stream);
/* Backward of the block above given dY (bf16 [B, L_out, C]) and the GELU' saved by the forward (dgelu_bf16, same layout;
 * NULL in the forward = inference, nothing saved); accumulates into dw [C, Cin, 10], dgamma, dbeta (fp32).
 * red_scratch: [B, 2 + Cin*10, C] fp64 workspace (fp64 atomics: the weight gradient is a difference of large sums).
 * The convolution itself runs on mma.sync tensor-core tiles in both directions (C must be 512). */
int wj_conv0_gn_gelu_bwd(const void* x_bf16, const float* w, const float* gamma, const float* beta, int B, int Cin,
                         int L, int C, int k, int stride, float eps, const double* moments, const float* stats,
                         const void* dy_bf16, const void* dgelu_bf16, void* red_scratch, float* dw, float* dgamma,
                         float* dbeta, void* stream);

/* LayerNorm over the last dim (D in {128,256,384,512,768,1024}), biased variance, one warp per row.
 * Writes any of: out_f32, out_bf16, stats [M,2] = (mean, rstd), rowsum [M,2] = (sum, sum of squares of the OUTPUT row).
 * Reference: nn.LayerNorm in nn.TransformerEncoderLayer (eps 1e-6, wavjepa/types/wavjepa_configs.py:38) and
 * feature_norms / encoder.norm / decoder.norm (eps 1e-5, wavjepa/jepa.py:109,127,130). */
int wj_layernorm_fwd(const void* x, int x_is_bf16, const float* gamma, const float* beta, float eps, int M, int D,
                     float* out_f32, void* out_bf16, float* stats, float* rowsum, void* stream);
/* dx (fp32 and/or bf16) from dy (fp32), the saved input x and stats; dgamma/dbeta (+=), colsum (+= sum_rows dx). */
int wj_layernorm_bwd(const float* dy, const void* x, int x_is_bf16, const float* stats, const float* gamma, int M,
                     int D, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta, float* colsum, void* stream);

/* Residual add + LayerNorm in one pass (post-norm layer, wavjepa/types/wavjepa_configs.py:29-47: x = LN(x + Linear(..))):
 * the row normalised is y = x (fp32 residual stream) + add (bf16 = the Linear output as autocast rounds it; NULL = 0).
 * The GEMM before it therefore writes 2 bytes per element and y never exists in HBM; outputs as wj_layernorm_fwd. */
int wj_add_layernorm_fwd(const float* x, const void* add_bf16, const float* gamma, const float* beta, float eps, int M,
                         int D, float* out_f32, void* out_bf16, float* stats, float* rowsum, void* stream);
/* Backward of the above.  Gradient w.r.t. the LayerNorm output = dy_f32 (fp32 residual branch, may be NULL) + dy_bf16
 * (bf16 data gradient of the Linear that consumed the output, may be NULL); y is re-formed as x + add_bf16. */
int wj_add_layernorm_bwd(const float* dy_f32, const void* dy_bf16, const float* x, const void* add_bf16,
                         const float* stats, const float* gamma, int M, int D, float* dx_f32, void* dx_bf16,
                         float* dgamma, float* dbeta, float* colsum, void* stream);

/* out[i] = (g*audio[clip, :, start_i : start_i+crop_len] - mean) / (std_unbiased + 1e-5), statistics over
 * (C, crop_len) jointly; i = clip*crops_per_clip + j; samples past clip_len read as zero; g = gain[clip] (NULL = 1).
 * JEPA.on_after_batch_transfer (wavjepa/jepa.py:291-311) and hear_api/runtime.py:12-16 (normalize). */
int wj_crop_norm(const float* audio, const int* starts, const float* gain, int n_clips, int channels,
                 int64_t clip_len, int crops_per_clip, int crop_len, void* out_bf16, float* out_f32, void* stream);
/* gain[clip] = 10^((target_dbfs - 20 log10(rms)) / 20) with rms over the whole clip (1 when rms == 0):
 * normalize_audio (hear_api/feature_helper.py:5-13). */
int wj_clip_gain(const float* audio, int n_clips, int channels, int64_t clip_len, float target_dbfs, float* gain,
                 void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * On-GPU input pipeline (data_modules/WebAudioDataModule.py:43-61, dataset_functions.py:92-114).
 * wj_resample_sinc: y[n*new + p] = sum_k table_t[k, p] * xpad[n*orig + k] (torchaudio's polyphase Kaiser-sinc
 *   resampler: conv1d with stride `orig` over x padded by (width, width + orig) zeros, K = 2*width + orig taps, `new`
 *   phases; orig/new already divided by their gcd; table_t is [K, new] fp32).  Outputs t < out_cap are stored, the
 *   rest of out[0:out_cap] is zero-filled (pad / crop to the fixed clip length); *sumsq (fp64, += ) receives the sum of
 *   squares of ALL target_length = ceil(new*length/orig) outputs (the RMS is taken before the crop).
 * wj_rms_gain_rows: clips[c, :] *= 10^((target_dbfs - 20 log10(sqrt(sumsq[c]/counts[c]))) / 20) (no-op when silent). */
int wj_resample_sinc(const float* x, int64_t length, const float* table_t, int orig, int new_, int width,
                     int64_t target_length, float* out, int64_t out_cap, double* sumsq, void* stream);
int wj_rms_gain_rows(float* clips, const double* sumsq, const int64_t* counts, int n_clips, int64_t row_len,
                     float target_dbfs, void* stream);

/* targets (=|+=) scale * instance_norm(x) with statistics over all T*D values of each instance (biased var, eps);
 * rowsum [B*T, 2] comes from wj_layernorm_fwd.  JEPA._make_targets (wavjepa/jepa.py:230-253). */
int wj_target_accum(const float* x, const float* rowsum, int B, int T, int D, float eps, float scale, int first,
                    float* inst_stats, float* targets, void* stream);

/* The same targets from all top-K layer outputs in one pass: xs / rowsums are HOST arrays of n_layers (<= 16) device
 * pointers (layer outputs [B*T, D] fp32 and their wj_layernorm_fwd rowsum [B*T, 2]); inst_stats: [n_layers, B, 2]
 * workspace.  targets = scale * sum_l instance_norm(x_l): every layer is read once, the targets written once. */
int wj_target_combine(const float* const* xs, const float* const* rowsums, int n_layers, int B, int T, int D, float eps,
                      float scale, float* inst_stats, float* targets, void* stream);

/* Variable-length multi-head attention over packed tokens: qkv bf16 [tokens, 3*D] (q|k|v), sequences given by
 * cu_seqlens [n_seqs+1], softmax(q k^T / sqrt(D/H)) v, head dim 32 or 64.  out bf16 [tokens, D];
 * lse2 fp32 [tokens, H] = log2-sum-exp2 of the scaled logits (saved for the backward; may be NULL).
 * total_tokens = rows of qkv.  Forward: sequences of <= 512 tokens run on tcgen05 (S = Q K^T and O = P V as UMMAs with
 * TMEM accumulators, P handed back through TMEM, softmax one query row per thread); longer ones on the mma.sync kernel.
 * Backward: head dim 32 with <= 128 tokens runs on tcgen05 (S, dP, dV, dK, dQ as UMMAs); everything else on mma.sync.
 * Reference: F.scaled_dot_product_attention with key_padding_mask inside nn.MultiheadAttention. */
int wj_attn_varlen_fwd(const void* qkv_bf16, const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D,
                       int H, void* out_bf16, float* lse2, void* stream);
int wj_attn_varlen_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16, const float* lse2,
                       const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D, int H,
                       void* dqkv_bf16, void* stream);

/* The same backward with the bias gradient of the in_proj Linear folded in: dbias[3 D] += column sums of dqkv.  On the
 * tcgen05 path (head dim 32, <= 128 tokens) the query third is reduced in the kernel's epilogue, the value third is added
 * as the column sums of dout (softmax rows sum to one: sum_k dV[k,:] = sum_q dO[q,:]) and the key third, which is
 * identically zero in exact arithmetic (softmax ignores a constant key shift), is left untouched; on the mma.sync path a
 * wj_colsum pass over the stored dqkv follows the kernel.  dbias may be NULL. */
int wj_attn_varlen_bwd_bias(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16, const float* lse2,
                            const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D, int H,
                            void* dqkv_bf16, float* dbias, void* stream);

/* wj_attn_varlen_bwd_bias that also takes head-dim-64 sequences of 385..400 tokens (the dense binaural WavJEPA-Nat
 * student of 2 x 200 tokens, fine-tuned through get_audio_representation): the per-query lse / delta then live in the
 * padding columns of the shared-memory Q rows, so the four 400-row tiles stay resident.  Shorter sequences take exactly
 * wj_attn_varlen_bwd_bias's kernels. */
int wj_attn_varlen_bwd_bias_long(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16, const float* lse2,
                                 const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D, int H,
                                 void* dqkv_bf16, float* dbias, void* stream);

/* Row gather: out[i, :] = src[idx[i], :] (idx NULL = identity, i.e. a cast); fp32 and/or bf16 outputs.
 * contextual_features[~ctx_masks] (wavjepa/jepa.py:399). */
int wj_gather_rows(const void* src, int src_is_bf16, const int* idx, int N, int D, float* out_f32, void* out_bf16,
                   void* stream);
/* out[idx[i], :] = src[i, :] (fp32): packed encoder rows back to their dense [B*T, D] positions
 * (JEPA.get_audio_representation, wavjepa/jepa.py:456-467). */
int wj_scatter_rows(const float* src, const int* idx, int N, int D, float* out, void* stream);
/* out_bf16[idx[i], :] = src[i, :] * h[idx[i], :] (h = the GELU' factors saved by an act == 1 GEMM epilogue; may be
 * NULL; idx NULL = identity); rows not listed are left untouched. */
int wj_scatter_dgelu(const float* src, const int* idx, const void* h_bf16, int N, int D, void* out_bf16, void* stream);

/* Predictor input: x0[r] = (vis_src[r] >= 0 ? ctx[vis_src[r]] : bf16(mask_token)) + pos[vis_pos[r]]
 * (JEPA.decoder_forward, wavjepa/jepa.py:425-435) and its backward (d_ctx fp32 [Nc, D] +=, d_mask_token [D] +=). */
int wj_predictor_assemble(const void* ctx_bf16, const float* mask_token, const float* pos, const int* vis_src,
                          const int* vis_pos, int N, int D, float* out_f32, void* out_bf16, void* stream);
int wj_predictor_assemble_bwd(const float* dx0, const int* vis_src, int N, int D, float* d_ctx, float* d_mask_token,
                              void* stream);
/* The context part of that backward as a gather with a fixed summation order (no atomics: the same bits in every run):
 * d_ctx[s] = sum over the G target groups, in order, of dx0[row of context row s in that group's predictor sequence];
 * written as fp32 and / or bf16 (either may be NULL).  ctx_vrow [Nc * G] int32 is workspace (the inverse of vis_src,
 * rebuilt by the call); cu_v [n_seqs + 1] are the predictor sequence offsets, n_seqs = B * G.  With this call
 * wj_predictor_assemble_bwd takes d_ctx = NULL and only accumulates the mask-token gradient. */
int wj_predictor_ctx_grad(const float* dx0, const int* vis_src, const int* cu_v, int n_seqs, int G, int Nc, int D,
                          int* ctx_vrow, float* d_ctx_f32, void* d_ctx_bf16, void* stream);

/* *loss += sum_i mean_d (pred[i,d] - targets[tgt_rows[i], d])^2 / (Nt + 1e-8); dpred (optional, bf16) = d loss / d pred.
 * JEPA.masked_loss (wavjepa/jepa.py:335-362) restricted to the target rows (all other rows have zero weight). */
int wj_masked_mse(const void* pred_bf16, const float* targets, const int* tgt_rows, int Nt, int D, float* loss,
                  void* dpred_bf16, void* stream);

/* Denoiser losses (wavjepa/denoiser.py:352-356): pred fp32 [2, M] = student features of the (clean, generated) halves,
 * target fp32 [M] = frozen-teacher features of the clean audio.  sums[h] (fp64, caller-zeroed) += sum (pred[h]-target)^2,
 * i.e. loss_clean = sums[0] / M, loss_denoise_dereverb = sums[1] / M; dpred (optional, fp32 [2, M]) = gradient of
 * alpha * loss_clean + (1 - alpha) * loss_denoise_dereverb. */
int wj_mse_pair(const float* pred, const float* target, int64_t M, float alpha, double* sums, float* dpred, void* stream);

/* Segmental-SNR mixing (data_modules/scene_module/generate_scenes_batch.py:107-146 add_noise): rows b of source / noise
 * [B, T] fp32; energies over the window [start_b, start_b + length_b); out = source + a_b * noise with
 * a_b = sqrt(E_source / (E_noise + 1e-9) * 10^(-snr_b / 10)).  energy: fp64 [B, 2] workspace. */
int wj_snr_mix(const float* source, const float* noise, const int* start, const int* length, const float* snr, int B,
               int64_t T, double* energy, float* out, void* stream);

/* teacher = teacher * decay + (1 - decay) * student, fp32, rounding exactly like
 * teacher.mul_(r).add_((1 - r) * student) (JEPA._step_teacher, wavjepa/jepa.py:193-198). */
int wj_ema_update(float* teacher, const float* student, int64_t n, double decay, void* stream);

/* *out (fp64) += sum (scale * x[i])^2 -- global gradient norm for clip_grad_norm_ (train.py:177-178). */
int wj_sumsq(const float* x, int64_t n, float scale, double* out, void* stream);
/* One fused multi-tensor AdamW step over a flat parameter buffer (torch.optim.AdamW semantics, wavjepa/jepa.py:215-222)
 * with the gradient scale (1/world_size) and clip coefficient min(1, max_norm / (sqrt(*grad_sumsq) + 1e-6)) folded in;
 * optionally refreshes the bf16 working copy of the weights. step is 1-based. */
int wj_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int step, float grad_scale, float max_norm, const double* grad_sumsq,
                  void* p_bf16, void* stream);
/* The same step with the EMA teacher update folded into the pass over the parameters (SURVEY.md 8(f)-1): for
 * i in [ema_lo, ema_hi): teacher[i - ema_lo] = teacher * ema_decay + (1 - ema_decay) * p_old[i] (the student value BEFORE
 * this optimizer step, as JEPA.training_step orders it, wavjepa/jepa.py:330-331) + its bf16 working copy. */
int wj_adamw_ema_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                      float eps, float weight_decay, int step, float grad_scale, float max_norm,
                      const double* grad_sumsq, void* p_bf16, float* teacher, void* teacher_bf16, int64_t ema_lo,
                      int64_t ema_hi, double ema_decay, void* stream);
int wj_cast_bf16(const float* x, void* y_bf16, int64_t n, void* stream);
/* a[i] += float(b[i]) (b bf16): joins an fp32 residual-branch gradient with a bf16 Linear data gradient. */
int wj_add_bf16(float* a, const void* b_bf16, int64_t n, void* stream);
/* out[n] += sum_m x[m, n] (bias gradients). */
int wj_colsum(const void* x, int x_is_bf16, int64_t M, int N, int64_t ld, float* out, void* stream);
int wj_scale_bf16(void* x_bf16, const float* scale_dev, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Reference-precision (TF32) inference path: the fp32 feature extraction of hear_api/runtime.py:98-145 with every GEMM
 * operand rounded to nearest tf32 (the tensor core truncates raw fp32, which doubles the error), fp32 accumulation,
 * exact erf GELU, fp32 residual stream.  Forward only.
 *
 * wj_gemm_tf32: out[b*L + t, n] = epilogue( sum_vc A(vc; t, b) * W[n, vc] ) with an fp32 operand A (wj_operand_t over
 *   4-byte elements: plain activations or the conv window views) and fp32 W [N, K] (leading dim ldw), both K-major,
 *   tcgen05.mma.kind::tf32.  K % 32 == 0, N % 128 == 0.  Epilogue: v = acc + bias; act 4: v = GELU_erf(v) (act 0: none);
 *   v += resid[row % resid_mod or row, n]; out = bf16(v), or fp32 v (rounded to nearest tf32 when round_out).
 *   accumulate / out2 / aux / out_rows / colsum must be unset. */
int wj_gemm_tf32(const wj_operand_t* A, const float* W, int64_t ldw, int L, int batch, int N, int K,
                 const wj_epilogue_t* epi, int round_out, void* stream);
/* Conv block 0 from fp32 input x [B, Cin, L] and unrounded fp32 weights: fp32 FMA on the CUDA cores, closed-form
 * GroupNorm statistics (moments / stats workspaces as wj_conv0_gn_gelu_fwd), exact erf GELU; out fp32 [B, L_out, C]
 * rounded to nearest tf32. */
int wj_conv0_gn_gelu_fwd_f32(const float* x, const float* w, const float* gamma, const float* beta, int B, int Cin,
                             int L, int C, int k, int stride, float eps, double* moments, float* stats, float* out,
                             void* stream);
/* Attention forward of wj_attn_varlen_fwd (bf16 qkv, Q/K/V and P on the tensor cores in bf16) writing O as fp32
 * [tokens, D] rounded to nearest tf32.  Head dim 64 and sequences of <= 512 tokens only; other shapes are refused. */
int wj_attn_varlen_fwd_f32out(const void* qkv_bf16, const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens,
                              int D, int H, float* out_f32, void* stream);
/* LayerNorm(x + add) with x fp32 and add fp32 (or NULL): out_f32 = the unrounded result, out_tf32 = the result rounded to
 * nearest tf32 (the next GEMM's operand); either may be NULL.  D as wj_layernorm_fwd. */
int wj_add_layernorm_fwd_f32(const float* x, const float* add_f32, const float* gamma, const float* beta, float eps,
                             int M, int D, float* out_f32, float* out_tf32, void* stream);
/* y[i] = x[i] rounded to nearest tf32 (y may be x). */
int wj_tf32_round(const float* x, float* y, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WAVJEPA_B200_H */
