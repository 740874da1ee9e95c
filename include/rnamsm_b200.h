/* rnamsm_b200 -- C ABI of the B200-native RNA-MSM forward path.
 *
 * Drop-in boundary.  The reference (yikunpku/RNA-MSM) is pure Python/PyTorch and has no FFI of
 * its own: the boundary it exposes for this path is the nn.Module API
 *   MSATransformer.forward(tokens, repr_layers, need_head_weights, return_contacts)  model.py:338-416
 *   AxialTransformerLayer.forward(x, self_attn_mask, self_attn_padding_mask, need_head_weights)
 *                                                                              modules.py:242-267
 *   RowSelfAttention.forward / ColumnSelfAttention.forward                     modules.py:802-821, 926-945
 *   FeedForwardNetwork.forward                                                 modules.py:423-427
 * plus the state-dict names and the two .npy outputs (RNA_MSM_Inference.py:150-166).
 * The Python package `rnamsm_b200` mirrors those classes one-for-one and binds the entry points
 * below with ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device unless named host_*;
 *   - no allocation inside: the caller (PyTorch) owns inputs, outputs and workspaces;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing syncs;
 *   - return value 0 = ok; non-zero = error, message in rnamsm_last_error() (thread-local);
 *   - `dtype` selects the arithmetic path: RNAMSM_F32 = fp32 FFMA kernels (parity path,
 *     <=1e-4 norm-relative vs the reference fp32 forward); RNAMSM_BF16 / RNAMSM_F16 = 16-bit
 *     operands on the tcgen05 tensor cores (kind::f16, same rate for both element types) with
 *     fp32 accumulation and an fp32 residual stream / LayerNorm / softmax (<=2e-2).  In the
 *     whole-layer drivers each attention block carries its own operand type
 *     (rnamsm_attn_weights.dtype).  Production precision is fp16 everywhere.  The optional "bf16"
 *     mode still runs the tied row-attention block in fp16: its logits are sums over R*64 products
 *     whose rounding errors add coherently on redundant MSAs (exported maps on the 2DRB_1 MSA:
 *     all-bf16 5.1e-2, bf16 with the fp16 row block 2.7e-2, fp16 5.4e-3; same tensor-core rate).
 *     There is no CPU fallback.
 *   - one MSA per call (B = 1): the reference never batches MSAs (RNA_MSM_Inference.py:147)
 *     and its tied-attention scaling depends on the padded row count (modules.py:713-715).
 *     rnamsm_msa_forward_batch runs several MSAs in one pass with exactly these per-MSA semantics.
 *   - activations are token-major: x[(r*C + c)*D + f], i.e. the reference's [R,C,B=1,D].
 */
#ifndef RNAMSM_B200_H_
#define RNAMSM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RNAMSM_ABI_VERSION 3

enum { RNAMSM_F32 = 0, RNAMSM_BF16 = 1, RNAMSM_F16 = 2 };
/* OR-ed into dtype RNAMSM_F32 for rnamsm_workspace_bytes / rnamsm_layer_forward / rnamsm_msa_forward: fp32 storage and
 * fp32 attention / LayerNorm / softmax as in the fp32 path, but the nn.Linear layers (88 % of the flops) run on the
 * tensor cores as rnamsm_linear_tf32 (three tf32 MMAs on hi / lo operand halves).  The tensor core accumulates its fp32
 * sums with truncation, so this mode is ~10x less exact per GEMM than the FFMA path (measured below) -- a fast
 * high-precision mode, not the <= 1e-4 parity path. */
#define RNAMSM_F32_TENSOR 0x100
#define RNAMSM_MAX_PEERS 8 /* GPUs of one NVSwitch box a single MSA can be sharded over */

/* Epilogues of rnamsm_linear. */
enum {
  RNAMSM_EPI_BIAS = 0,          /* out = x W^T + b          (out in compute dtype)                 */
  RNAMSM_EPI_BIAS_GELU = 1,     /* out = gelu_erf(x W^T + b)  nn.GELU(), modules.py:416,424        */
  RNAMSM_EPI_BIAS_RESIDUAL = 2  /* out(fp32) += x W^T + b     NormalizedResidualBlock, modules.py:397 */
};

int rnamsm_version(void);
const char* rnamsm_last_error(void);
/* 0 when the current device is a compute-capability 10.x part (B200); error otherwise. */
int rnamsm_device_check(void);
/* Number of kernels this library has launched in the calling process (bench.py gpu_launches). */
long long rnamsm_launch_count(void);

/* CTA pairs (clusters of 2) the persistent tcgen05 GEMM grid uses on this device: the number
 * that can be co-resident (cudaOccupancyMaxActiveClusters), known after the first 16-bit launch;
 * 0 before. */
int rnamsm_gemm_pairs(void);

/* Optional device timing of every kernel launch by class (cudaEvents recorded on the launching
 * stream around each launch).  enable(1) resets and starts recording, enable(0) stops;
 * collect() synchronises the recorded events and returns the accumulated milliseconds and launch
 * counts per class (arrays of rnamsm_profile_num_classes() entries).  Host-side, not thread-safe. */
int rnamsm_profile_enable(int on);
int rnamsm_profile_num_classes(void);
const char* rnamsm_profile_class_name(int cls);
int rnamsm_profile_collect(double* ms_out, long long* launches_out, int n);

/* K1 -- token + learned-position + per-row scalar embedding, LayerNorm, pad zeroing.
 * Replaces model.py:346-367 and LearnedPositionalEmbedding.forward (modules.py:286-300).
 * tokens [R,C] int64; tok_emb [vocab,D]; pos_emb [n_pos,D]; row_pos [>=R] scalars or NULL;
 * x_out [R*C, D] fp32; pad_out [R*C] uint8 (1 where token == pad_idx) or NULL. */
int rnamsm_embed_layernorm(const int64_t* tokens, int R, int C, const float* tok_emb, int vocab,
                           const float* pos_emb, int n_pos, const float* row_pos, const float* ln_w,
                           const float* ln_b, int D, int pad_idx, float eps, float* x_out,
                           uint8_t* pad_out, void* stream);

/* K2 / K9 -- LayerNorm over the last dim (nn.LayerNorm(D), biased variance), fp32 in,
 * fp32 / bf16 / fp16 out (modules.py:382,387; model.py:331-332,396).  tr_R, tr_C > 0 (with
 * tr_R * tr_C == n_rows) additionally permutes the tokens from token-major (r * C + c) to
 * column-major (c * R + r) order on the way out -- the layout the column-attention block works in;
 * 0, 0 keeps the order. */
int rnamsm_layernorm(const float* x, const float* w, const float* b, void* y, int y_dtype, long long n_rows,
                     int D, float eps, int tr_R, int tr_C, void* stream);

/* K3 / K6-out / K8 -- nn.Linear with fused epilogue: out = epi(x[M,K] W[N,K]^T + bias[N]).
 * x, W in `dtype`.  For RNAMSM_EPI_BIAS: columns [0,q_cols) are multiplied by q_scale after the
 * bias (q *= scaling, modules.py:766, 905) and, when row_mask != NULL, by (1 - row_mask[m])
 * (padded query rows zeroed, modules.py:767-772).  `out` is in `dtype` except for
 * RNAMSM_EPI_BIAS_RESIDUAL where it is the fp32 residual stream updated in place (16-bit path: by TMA
 * reduce-add, so `out` must not be read or written by anything else on the stream meanwhile).
 * 16-bit path: N, K and q_cols multiples of 64; any M (tails are clipped by the TMA unit). */
int rnamsm_linear(const void* x, const void* W, const float* bias, long long M, int N, int K, int dtype,
                  int epilogue, float q_scale, int q_cols, const uint8_t* row_mask, void* out, void* stream);

/* K4 -- tied row-attention logits (modules.py:774): for every head h
 *   partial[s][h][i][j] = sum_{r in split s} sum_d q[r,i,h,d] k[r,j,h,d]
 * qkv [R*C, 3*H*64] in `dtype`, q|k|v packed along the feature dim, q already scaled.
 * partial: fp32 [n_splits, H, C, C].  n_splits >= 1 row ranges are summed by K5. */
int rnamsm_row_attn_logits(const void* qkv, int R, int C, int H, int dtype, float* partial, int n_splits,
                           void* stream);
/* fp32 nn.Linear on the tensor cores (the fp32 path's route inside rnamsm_layer_forward / rnamsm_msa_forward): both fp32
 * operands are split on the device into a tf32 "hi" part and an exact fp32 remainder "lo", and every k-step issues three
 * tcgen05.mma kind::tf32 into one fp32 accumulator (hi*hi + lo*hi + hi*lo): near-fp32 results (the operand split is
 * exact to 2^-23; what remains is the tensor core's truncating fp32 accumulation, norm-relative error a few 1e-6,
 * tests/test_gpu_ops.py) at 8x the FFMA kernel's rate (300 vs 37 TFLOP/s measured).  Same epilogues as rnamsm_linear with
 * dtype RNAMSM_F32 (out fp32 [M, N]; residual: in place).  scratch: rnamsm_linear_tf32_scratch_bytes(M, N, K) device
 * bytes, 256 B aligned.  N and K multiples of 32. */
size_t rnamsm_linear_tf32_scratch_bytes(long long M, int N, int K);
int rnamsm_linear_tf32(const float* x, const float* W, const float* bias, long long M, int N, int K, int epilogue,
                       float q_scale, int q_cols, const uint8_t* row_mask, float* out, void* scratch, size_t scratch_bytes,
                       void* stream);

/* NormalizedResidualBlock (modules.py:385-401) in one kernel, 16-bit path: resid[M, N] (fp32, in place) += x[M, K] W[N, K]^T
 * + bias, and y[M, N] (16-bit, y_dtype) = LayerNorm(resid) * ln_w + ln_b over the N features of each finished row --
 * the operand of the next block's first GEMM, so no stand-alone LayerNorm pass reads the stream again.  The CTA whose
 * TMA reduce-adds complete a 128-row block (arrivals counted in `counters`) reads the rows back from L2 and normalises.
 * N % 128 == 0, N <= 1024.  tr_R, tr_C > 0: y row (m % tr_C) * tr_R + m / tr_C (column-major token order).
 * counters: device int32 [2 * ceil(M / 256)], ZERO on entry; the kernel leaves them zero again (reusable as is). */
int rnamsm_linear_residual_layernorm(const void* x, const void* W, const float* bias, long long M, int N, int K, int dtype,
                                     float* resid, const float* ln_w, const float* ln_b, float eps, void* y, int y_dtype,
                                     int tr_R, int tr_C, int* counters, void* stream);

/* K4 + K5 + K6 in ONE launch for short alignments (C <= 128), 16-bit dtypes only: tied logits per (head, row chunk) ->
 * grid barrier -> softmax with key mask (fp32 map into probs_out [H,C,C], 16-bit rows into probs_lp [H,C,ld_lp]) ->
 * grid barrier -> ctx [R*C, H*64] = P V (modules.py:752-821).  A cooperative launch of H x n_chunks CTAs; this is the
 * route rnamsm_layer_forward / rnamsm_msa_forward / rnamsm_msa_forward_batch take whenever
 * rnamsm_row_attn_short_chunks(R, C, H) > 0 (it returns 0 for C > 128 or with RNAMSM_ROW_SHORT=0 in the environment).
 * partial: fp32 scratch [n_chunks, H, C, C]; n_chunks as returned by rnamsm_row_attn_short_chunks (any value with
 * H * n_chunks <= #SMs and no empty chunk is accepted).  Split sums are taken in a fixed order: results do not
 * depend on timing. */
int rnamsm_row_attn_short_chunks(int R, int C, int H);
int rnamsm_row_attn_short(const void* qkv, int R, int C, int H, int dtype, const uint8_t* key_pad, float logit_scale,
                          float* partial, int n_chunks, float* probs_out, void* probs_lp, int ld_lp, void* ctx,
                          void* stream);

/* Suggested split count for K4: as many row ranges as fit ONE wave of the launch (74 CTA pairs in the
 * 16-bit path), at least 8 rows each. */
int rnamsm_row_attn_splits(int R, int C, int H, int dtype);

/* K5 -- sum the split partials, multiply by logit_scale (1 when q already carries the whole
 * align_scaling; 1/sqrt(R) in the 16-bit path where q carries only 64^-1/2), mask keys
 * (logit = -10000 where key_pad[j], modules.py:780-784), softmax over j (modules.py:818).  probs_out fp32 [H,C,C] is the exported attention map
 * (written straight into the caller's [N,H,C,C] slab); probs_lp ([H,C,ld_lp] in `dtype`, columns
 * >= C zero-filled) feeds K6 and may be NULL in fp32 mode where K6 reads probs_out. */
int rnamsm_row_softmax(const float* partial, int n_splits, int H, int C, const uint8_t* key_pad, float logit_scale,
                       float* probs_out, void* probs_lp, int ld_lp, int dtype, void* stream);

/* K6 -- ctx[r,i,h,:] = sum_j P[h,i,j] v[r,j,h,:] (modules.py:797).  probs [H,C,ldp] in `dtype`;
 * ctx [R*C, H*64] in `dtype`. */
int rnamsm_row_attn_av(const void* probs, int ldp, const void* qkv, int R, int C, int H, int dtype, void* ctx,
                       void* stream);

/* K7 -- column attention over the MSA depth, flash-style (modules.py:896-923): for every column c
 * and head h, ctx[i,c,h,:] = softmax_j(q[i,c,h,:].k[j,c,h,:]) v[j,c,h,:]; q already scaled by
 * 64^-0.5; keys with pad[j*C+c] != 0 get logit -10000 (modules.py:911-915).  R >= 2 (the R == 1
 * shortcut of modules.py:882-894 is handled by the caller as out_proj(v_proj(x))).
 * qkv_col_major = 0: q|k|v is token-major [R, C, 3D] like every other activation;
 * qkv_col_major = 1 (16-bit path only): q|k|v is [C, R, 3D], i.e. produced from a LayerNorm output
 * written with tr_R / tr_C -- the rows a (column, head) problem reads are then 3D elements apart
 * instead of C * 3D, which is what lets the TMA unit stream K/V (see DESIGN.md).  pad and ctx are
 * token-major ([R*C] and [R*C, D]) in both cases. */
int rnamsm_col_attn(const void* qkv, int R, int C, int H, int dtype, int qkv_col_major, const uint8_t* pad, void* ctx,
                    void* stream);

/* Column-attention probabilities of K7 on request (the reference's [H, C, B, R, R] for one MSA, modules.py:907-918):
 * from the same q|k and pad as rnamsm_col_attn (either q|k layout; the column-major one in the 16-bit path only),
 *   probs_out fp32 [H, C, R, R]: P[h,c,i,j] = softmax_j(q[i,c,h,:].k[j,c,h,:]), logit -10000 where pad[j*C+c] != 0;
 *   mean_out  fp32 [H, R, R]:    (1/C) sum_c P[h,c,i,j] over every column, computed without the full tensor.
 * Either output may be NULL.  R == 1 gives all ones (modules.py:882-894; q|k and scratch are not read).
 * scratch: rnamsm_col_probs_scratch_bytes(R, C, H) device bytes (per-row max and log-sum).  dtype RNAMSM_F32 runs FFMA
 * kernels (expf), the 16-bit dtypes tcgen05 (ex2.approx).  Deterministic: no atomics, columns summed in order. */
int rnamsm_col_attn_probs(const void* qkv, int R, int C, int H, int dtype, int qkv_col_major, const uint8_t* pad,
                          float* probs_out, float* mean_out, void* scratch, void* stream);

/* K9b -- tied LM-head projection logits[m, v] = h[m,:] . E[v,:] + bias[v] (modules.py:318), fp32. */
int rnamsm_vocab_proj(const float* h, const float* E, const float* bias, long long M, int V, int D, float* out,
                      void* stream);

/* Contact head (SURVEY.md 8f row 2) -- ContactPredictionHead.forward, modules.py:347-366 with
 * utils/tensor.py:98-113: over the L x L block [start, start+L)^2 of each of the K = layers*heads maps
 * (maps fp32 [K, C, C]; start = 1 strips BOS, model.py:412-414): symmetrize, average-product correction,
 * then sigmoid(bias + sum_k w[k] * .) -> out fp32 [L, L].  workspace: K*L + K floats. */
int rnamsm_contact_head(const float* maps, int K, int C, int start, int L, const float* w, const float* bias,
                        float* out, float* workspace, void* stream);

/* SS-predictor input packing (SURVEY.md 8f row 3): _downstream_tasks/SS/code/pre_processing/data_processing.py:32-48
 * + data_fomat.py:38-59 from the device-resident maps: out fp32 [8 + K, L, L] (= x[0] of the [1,128,L,L] input):
 * channels 0-3 one-hot of seq[i] over A,C,G,U, 4-7 one-hot of seq[j], 8.. = map k over the block
 * [start, start+L)^2.  seq_codes uint8 [L]: 0..3 = A,C,G,U, anything else = unknown (all-zero one-hot). */
int rnamsm_ss_pack(const float* maps, int K, int C, int start, int L, const uint8_t* seq_codes, float* out, void* stream);

/* RSA-predictor input packing (SURVEY.md 8f row 4): _downstream_tasks/RSA/predict.py:131-141 from the
 * device-resident hidden states: out fp32 [n_oh + D + 1, L] (= x_train[0] after its transpose):
 * channels 0-3 = (one-hot(seq[i] over A,C,G,U) - mu_oh) / std_oh evaluated in float64 as the reference
 * does, then D channels (emb[i, f] - mu_emb[f]) / std_emb[f] in fp32, then a channel of ones.
 * emb: row i at emb + i*ld (pass the final x of rnamsm_msa_forward offset past BOS, ld = D).
 * mu_oh / std_oh: HOST arrays of 4 doubles, or both NULL for the embedding-only predictor (n_oh = 0,
 * models/RNA-MSM_Emb).  mu_emb / std_emb: device fp32 [D].  seq_codes as for rnamsm_ss_pack.
 * Bit-identical to the reference's numpy expression. */
int rnamsm_rsa_pack(const float* emb, int ld, int L, int D, const uint8_t* seq_codes, const double* mu_oh,
                    const double* std_oh, const float* mu_emb, const float* std_emb, float* out, void* stream);

/* ---- MSA ingest (SURVEY.md 8f row 1): the step in front of the hot path, on the device ---------------
 * rnamsm_msa_clean: MSA.from_fasta's character rules (utils/align.py:311-313) as a per-row compaction.
 *   raw = the record bodies back to back (newlines allowed), offsets [N+1] (int64) delimit record n;
 *   chars_out uint8 [N, L]; *bad_row (device int) = 1 + index of a row whose cleaned length != L, else 0.
 * rnamsm_msa_greedy_select: MSA.greedy_select (utils/align.py:128-148; sample_method "diversity-max" /
 *   "diversity-min"): selected_out (device int32 [num]) = the sorted row indices, identical to the reference's
 *   including how exact ties fall (its float64 mean is reproduced operation for operation: numpy's pairwise
 *   sum over the picks, then / k, first index on equal values).  1 <= num <= min(N, 1024).
 *   workspace: rnamsm_msa_greedy_workspace(N, num) bytes (N * (num-1) uint16 mismatch counts + scratch).
 * rnamsm_msa_tokenize: Vocab.encode (utils/tokenization.py:107-129) of the selected rows (rows may be NULL
 *   = all rows in order): tokens_out int64 [R, L+1], column 0 = bos, the input of rnamsm_msa_forward. */
int rnamsm_msa_clean(const uint8_t* raw, const long long* offsets, int N, int L, uint8_t* chars_out, int* bad_row,
                     void* stream);
size_t rnamsm_msa_greedy_workspace(int N, int num);
int rnamsm_msa_greedy_select(const uint8_t* chars, int N, int L, int num, int want_max, int* selected_out,
                             void* workspace, void* stream);
int rnamsm_msa_tokenize(const uint8_t* chars, int L, const int* rows, int R, const uint8_t* lut256, int bos,
                        int64_t* tokens_out, void* stream);

/* ---- whole-layer / whole-model drivers (same kernels, one call) ------------------------------ */

typedef struct rnamsm_attn_weights {
  const float* ln_w; /* [D] pre-LN of the NormalizedResidualBlock */
  const float* ln_b;
  const void* w_qkv; /* [3D, D] rows = q_proj | k_proj | v_proj, compute dtype */
  const float* b_qkv; /* [3D] */
  const void* w_out; /* [D, D] compute dtype */
  const float* b_out; /* [D] */
  int dtype;          /* operand type of w_qkv / w_out and of this block's arithmetic: RNAMSM_BF16 or
                         RNAMSM_F16 in the 16-bit path (0 = same as the call's dtype); ignored (fp32)
                         when the call's dtype is RNAMSM_F32 */
} rnamsm_attn_weights;

typedef struct rnamsm_layer_weights {
  rnamsm_attn_weights row; /* layers.{l}.row_self_attention.*    */
  rnamsm_attn_weights col; /* layers.{l}.column_self_attention.* */
  const float* ffn_ln_w;
  const float* ffn_ln_b;
  const void* fc1_w; /* [F, D] */
  const float* fc1_b;
  const void* fc2_w; /* [D, F] */
  const float* fc2_b;
} rnamsm_layer_weights;

typedef struct rnamsm_model_weights {
  int num_layers, embed_dim, num_heads, ffn_dim, vocab, n_pos, pad_idx;
  float ln_eps;
  const float* tok_emb;  /* embed_tokens.weight [vocab, D] */
  const float* pos_emb;  /* embed_positions.weight [n_pos, D] */
  const float* row_pos;  /* msa_position_embedding flattened [1024] or NULL */
  const float* ln_before_w;
  const float* ln_before_b;
  const float* ln_after_w;
  const float* ln_after_b;
  const float* lm_dense_w; /* [D, D] fp32 (fp32 path, and the 16-bit path when lm_dense_w16 is NULL) */
  const float* lm_dense_b;
  const float* lm_ln_w;
  const float* lm_ln_b;
  const float* lm_bias;   /* [vocab] */
  const rnamsm_layer_weights* layers; /* host array, num_layers entries */
  const void* lm_dense_w16; /* [D, D] in the call's 16-bit dtype, or NULL: the LM head's dense GEMM on the tensor cores */
} rnamsm_model_weights;

/* Bytes of scratch rnamsm_layer_forward / rnamsm_msa_forward need for an R x C MSA. */
size_t rnamsm_workspace_bytes(int R, int C, int D, int H, int F, int dtype);
/* Scratch of rnamsm_col_attn_probs, and what rnamsm_layer_forward_col_probs / rnamsm_msa_forward_col_probs need on top
 * of their usual workspace when they export column probabilities: two fp32 [H, C, R], 256 B aligned; 0 for an empty shape. */
size_t rnamsm_col_probs_scratch_bytes(int R, int C, int H);

/* Range diagnostics for the 16-bit path.  rnamsm_range_scan: counters[0] += number of elements of buf (16-bit, n
 * elements) that are non-finite or sit at the largest finite value of the type (where the kernels' cvt.rn.satfinite
 * clamps: 65504 for fp16), counters[1] = max(counters[1], float bits of the largest |v| below that).  counters: two
 * uint64 on the device, zeroed by the caller.  rnamsm_debug_range_watch(counters): while non-NULL, rnamsm_layer_forward /
 * rnamsm_msa_forward scan every 16-bit activation they write (LayerNorm outputs, q|k|v, attention contexts, post-GELU
 * hidden) into those counters -- a debugging aid for checkpoints whose activations might leave the fp16 range (then
 * use precision "bf16"); NULL switches it off (default; process-wide, not thread-safe). */
int rnamsm_range_scan(const void* buf, long long n, int dtype, unsigned long long* counters, void* stream);
int rnamsm_debug_range_watch(unsigned long long* counters);

/* One AxialTransformerLayer (modules.py:242-267) in place on x [R*C, D] fp32.
 * pad [R*C] uint8 or NULL.  row_probs_out [H,C,C] fp32 or NULL (then a scratch map is used).
 * With LayerNorm fusion enabled (RNAMSM_FUSE_LN=1, 16-bit path; off by default -- it is exact but measured slower than
 * the stand-alone pass, see csrc/api.cu) every residual GEMM of the layer also emits the LayerNorm its successor consumes.
 * To chain layers without any stand-alone LayerNorm: pass the NEXT layer's row-block LayerNorm as next_ln_w / next_ln_b
 * (next_ln_dtype = that block's operand type, 0 = inherit `dtype`) -- this call's fc2 epilogue then leaves
 * LayerNorm(x) in the workspace -- and call the next layer with xn_ready = 1 on the SAME workspace.  xn_ready = 0 and
 * next_ln_w = NULL is the self-contained form.  rnamsm_fused_layernorm(dtype) tells whether the chain is available
 * (16-bit dtype and RNAMSM_FUSE_LN=1); otherwise xn_ready / next_ln_* must be 0 / NULL. */
int rnamsm_fused_layernorm(int dtype);
int rnamsm_layer_forward(const rnamsm_layer_weights* w, int D, int H, int F, float ln_eps, float* x, int R, int C,
                         const uint8_t* pad, int dtype, float* row_probs_out, void* workspace,
                         size_t workspace_bytes, int xn_ready, const float* next_ln_w, const float* next_ln_b,
                         int next_ln_dtype, void* stream);
/* rnamsm_layer_forward that also exports the column attention's probabilities: col_probs_out fp32 [H, C, R, R] and / or
 * col_mean_out fp32 [H, R, R] (as rnamsm_col_attn_probs; NULL = not wanted).  With either set, workspace_bytes must
 * cover rnamsm_workspace_bytes(...) + rnamsm_col_probs_scratch_bytes(R, C, H).  Both NULL: same launches, same
 * results as rnamsm_layer_forward. */
int rnamsm_layer_forward_col_probs(const rnamsm_layer_weights* w, int D, int H, int F, float ln_eps, float* x, int R, int C,
                                   const uint8_t* pad, int dtype, float* row_probs_out, float* col_probs_out,
                                   float* col_mean_out, void* workspace, size_t workspace_bytes, int xn_ready,
                                   const float* next_ln_w, const float* next_ln_b, int next_ln_dtype, void* stream);

/* MSATransformer.forward (model.py:338-416) for one MSA.
 *   tokens [R,C] int64 -> x (caller-provided fp32 [R*C, D] buffer; holds the final
 *   emb_layer_norm_after output on return), row_attn_out [N,H,C,C] fp32 or NULL,
 *   rep_out: host array of num_layers+1 device pointers (or NULL entries): rep_out[l] receives a
 *   copy of the hidden state after l layers for l < N (model.py:393-394); entry N is ignored
 *   (x itself is representation N).  logits_out [R*C, vocab] fp32 or NULL (LM head skipped).
 *   has_pad: 0 = the caller knows there is no <pad> token (padding_mask None, model.py:347-348). */
int rnamsm_msa_forward(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                       float* x, float* row_attn_out, float* const* rep_out, float* logits_out, void* workspace,
                       size_t workspace_bytes, void* stream);
/* rnamsm_msa_forward that also exports every layer's column-attention probabilities: col_probs_out fp32
 * [N, H, C, R, R] and / or col_mean_out fp32 [N, H, R, R] (NULL = not wanted).  With either set, workspace_bytes must
 * cover what rnamsm_msa_forward needs plus rnamsm_col_probs_scratch_bytes(R, C, H).  Both NULL: same launches, same
 * results as rnamsm_msa_forward. */
int rnamsm_msa_forward_col_probs(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                 int dtype, float* x, float* row_attn_out, float* col_probs_out, float* col_mean_out,
                                 float* const* rep_out, float* logits_out, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* Several short MSAs in one pass (SURVEY.md 8f row 4).  tokens: the int64 grids back to back
 * ([R[0]*C[0]] then [R[1]*C[1]] ...); R, C, has_pad: HOST arrays of n_msa entries (has_pad may be NULL);
 * x: fp32 [sum R*C, D], holds every MSA's final hidden states in the same order on return;
 * row_attn_out: HOST array of n_msa device pointers ([N,H,C[i],C[i]] fp32 each; NULL array or NULL entries
 * = not wanted).  The token-local steps (LayerNorms, the six projections / FFN GEMMs per layer) run once
 * over all tokens; the tied row attention and the column attention run per MSA with that MSA's own
 * 1/sqrt(R[i]) (modules.py:713-715), so each MSA's results are bit-identical to its own
 * rnamsm_msa_forward call -- this is NOT the reference's padded [B,R,C] batch.  16-bit dtypes, R[i] >= 2. */
size_t rnamsm_batch_workspace_bytes(int n_msa, const int* R, const int* C, int D, int H, int F, int dtype);
int rnamsm_msa_forward_batch(const rnamsm_model_weights* m, int n_msa, const int64_t* tokens, const int* R, const int* C,
                             const uint8_t* has_pad, int dtype, float* x, float* const* row_attn_out, void* workspace,
                             size_t workspace_bytes, void* stream);

/* Masked marginals of the LM head for one MSA (pseudo-log-likelihood, zero-shot mutant scores; utils/likelihood.py).
 * Entry k of the outputs is computed on `tokens` [R, C] with token (row, cols[k]) replaced by mask_idx: the LM-head
 * logits at (row, cols[k]) into logits_out [n_cols, vocab] (NULL = not wanted) and their log_softmax into
 * logprobs_out [n_cols, vocab].  mask_idx < 0: nothing is masked, one forward, every listed column read from it.
 * cols: DEVICE int32 [n_cols]; an entry that is out of range or names a <pad> token of `row` gives a NaN row in both
 * outputs.  dtype: as rnamsm_msa_forward (RNAMSM_F32_TENSOR included).  16-bit with R >= 2: the masked grids run in
 * passes of `group` through the layer path of rnamsm_msa_forward_batch; otherwise one forward per grid.  Only the scored
 * token of each grid goes through the final LayerNorm and the LM head.  The logits are bit-identical to
 * rnamsm_msa_forward's logits of the masked grid at that token.  workspace: rnamsm_score_workspace_bytes(..., group)
 * bytes, 256 B aligned; `group` sizes it (0 = invalid arguments). */
size_t rnamsm_score_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group);
int rnamsm_msa_masked_marginals(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                int dtype, int row, const int* cols, int n_cols, int mask_idx, int group,
                                float* logits_out, float* logprobs_out, void* workspace, size_t workspace_bytes,
                                void* stream);

/* Sequences generated from one MSA by iterative masked sampling with the LM head.  n_chains chains start from
 * `tokens` [R, C] (NULL: from the states already in tokens_out, to resume a run) and take steps start_step ..
 * start_step + steps - 1.  Step s of chain k masks token (r, c) when r is in `rows`, c >= 1, the token is not <pad> and
 * u_mask(seed, k, s, r, c) < mask_prob; runs the masked grid through the forward; runs the final LayerNorm and the LM
 * head on the `rows` only; and replaces each masked token by a draw from softmax(logits / temperature) over the tokens
 * of allowed_bitmask (bit v = vocabulary entry v; not <pad>, not <mask>, which is the last vocabulary entry) by inverse
 * CDF with u_draw(seed, k, s, r, c); temperature 0 takes the argmax, ties to the lowest index.  The uniforms are
 * Philox4x32-10 with key (seed low, seed high) and counter (k, s, r * C + c, 0 = mask | 1 = draw), u = (word0 >> 8) *
 * 2^-24 (csrc/sample.cu), so a result depends on none of group, the call split of the steps or the GPU.  rows: DEVICE
 * int32 [n_rows], ascending and distinct, in [0, R).  tokens_out: int64 [n_chains, R, C], the chains' final states.
 * dtype: as rnamsm_msa_forward (RNAMSM_F32_TENSOR included).  16-bit with R >= 2: `group` chains per pass through the
 * layer path of rnamsm_msa_forward_batch; otherwise one forward per grid.  Enqueues only: no synchronisation, no
 * allocation.  workspace: rnamsm_sample_workspace_bytes(..., group, n_rows) bytes, 256 B aligned (0 = invalid
 * arguments). */
size_t rnamsm_sample_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group, int n_rows);
int rnamsm_msa_gibbs_sample(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                            const int* rows, int n_rows, int n_chains, int steps, int start_step, float mask_prob,
                            float temperature, unsigned allowed_bitmask, unsigned long long seed, int group,
                            int64_t* tokens_out, void* workspace, size_t workspace_bytes, void* stream);

/* Categorical Jacobian of the LM head for one query row (Zhang et al., PNAS 2024): how the logits of every listed
 * residue move when one residue is substituted.  With G(i, a) = `tokens` [R, C] with token (row, positions[i]) replaced
 * by alphabet[a], and f(G)[j, b] the LM-head logit of G at (row, positions[j]) for token alphabet[b]:
 *   jacobian_out[i, a, j, b] = f(G(i, a))[j, b] - f(tokens)[j, b]        fp32 [P, A, P, A]
 * Only the slabs listed in `entries` run (one forward each, plus one of `tokens`); every other slab is exactly 0 --
 * callers list every (i, a) whose alphabet[a] differs from the wild type at positions[i].  positions: HOST int32 [P],
 * grid columns; alphabet: HOST int32 [A], vocabulary indices; entries: HOST int32 [n_entries], the slabs i * A + a,
 * strictly ascending.  They are staged into the workspace with one cudaMemcpyAsync.  dtype: as rnamsm_msa_forward
 * (RNAMSM_F32_TENSOR included).  16-bit with R >= 2: `group` grids per pass through the layer path of
 * rnamsm_msa_forward_batch; otherwise one forward per grid.  Only the query row of each grid goes through the final
 * LayerNorm and the LM head, so each slab is bit-identical to the difference of rnamsm_msa_forward's logits.  Enqueues
 * only: no synchronisation, no allocation.  workspace: rnamsm_jacobian_workspace_bytes(..., group, P, A, n_entries)
 * bytes, 256 B aligned (0 = invalid arguments). */
size_t rnamsm_jacobian_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group, int P, int A,
                                       int n_entries);
int rnamsm_msa_categorical_jacobian(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                    int dtype, int row, const int* positions, int P, const int* alphabet, int A,
                                    const int* entries, int n_entries, int group, float* jacobian_out, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* Contact map [P, P] fp32 from a categorical Jacobian J [P, A, P, A] (csrc/jacobian.cu): centre J over each of its four
 * axes in turn (i, a, j, b), F[i, j] = Frobenius norm of the centred A x A block (i, j) with F[i, i] = 0, average
 * product correction F - rowsum colsum^T / total (0 when total == 0) with the diagonal zeroed again, and
 * (F + F^T) / 2.  Fixed-order float64 reductions, no atomics: bitwise reproducible.  scratch:
 * rnamsm_jacobian_contacts_scratch_bytes(P, A) bytes, 256 B aligned (8 (P A)^2 + 8 P^2 + small). */
size_t rnamsm_jacobian_contacts_scratch_bytes(int P, int A);
int rnamsm_jacobian_contacts(const float* J, int P, int A, float* contacts_out, void* scratch, size_t scratch_bytes,
                             void* stream);

/* Full-length features of an alignment longer than the learned column positions, from overlapping windows
 * (csrc/windows.cu).  tokens [R, C] with BOS at column 0, L = C - 1 residues, no EOS.  W = min(window, L); window k
 * starts at residue s_k = min(k * stride, L - W), k < K = 1 + ceil((L - W) / stride), and is the grid [R, W + 1] of
 * column 0 and columns 1 + s_k .. W + s_k, run as an MSA of its own.
 * rnamsm_window_starts: the one implementation of that plan.  Returns K and writes s_0 .. s_{K-1} to HOST starts_out
 * (when not NULL); 0 for invalid arguments (L < 1, or not 1 <= stride <= window), with the reason in rnamsm_last_error.
 * rnamsm_msa_forward_windows: each window's row 0 of the final representation and its N*H row-attention maps (and, with
 * contacts_out, its contact-head map with regression weights contact_w [N*H] and contact_b [1] or NULL), BOS stripped,
 * stitched with tent weights w_k(p) = min(p - s_k + 1, s_k + W - p):
 *   emb_out [L, D]          emb[p] = sum_k c_k(p) emb_k[p - s_k],  c_k(p) = w_k(p) / sum_k' w_k'(p)
 *   atp_out [N*H, L, L]     atp[h, i, j] = sum_k c_k(i, j) map_k[h, i - s_k, j - s_k] over the windows holding i and j,
 *                           c_k(i, j) = w_k(i) w_k(j) / sum_k' w_k'(i) w_k'(j); exactly 0 where no window holds both
 *   contacts_out [L, L]     as atp, or NULL
 * Coefficients: float64 quotients of the integer sums rounded once to fp32; fp32 sums acc = fmaf(c_k, v_k, acc) from 0 in
 * ascending k, so the outputs do not depend on `group`, and an entry one window covers is that window's value bit for
 * bit.  Every output element is written (no clearing needed).  window <= n_pos - pad_idx - 2 (the learned positions).
 * dtype: as rnamsm_msa_forward (RNAMSM_F32_TENSOR included); the windows run `group` per pass on the route of
 * rnamsm_msa_masked_marginals (16-bit with R >= 2: the batch layer path; otherwise one forward per grid).  has_pad: the
 * input holds pad tokens (a window without any gives the same bits either way).  Enqueues only: no synchronisation, no
 * allocation.  workspace: rnamsm_windows_workspace_bytes(R, C, D, H, F, N layers, dtype, group, window, stride,
 * contacts wanted) bytes, 256 B aligned (0 = invalid arguments). */
int rnamsm_window_starts(int L, int window, int stride, int* starts_out);
size_t rnamsm_windows_workspace_bytes(int R, int C, int D, int H, int F, int N, int dtype, int group, int window, int stride,
                                      int want_contacts);
int rnamsm_msa_forward_windows(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                               int window, int stride, int group, float* emb_out, float* atp_out, float* contacts_out,
                               const float* contact_w, const float* contact_b, void* workspace, size_t workspace_bytes,
                               void* stream);

/* Statistics of an alignment itself, with no model (csrc/coevolution.cu; Morcos et al., PNAS 2011).  tokens: int64
 * [N, C] as rnamsm_msa_tokenize writes them, column 0 BOS, residues 1 .. L = C - 1, N >= 1, L >= 1.  States: A G C U
 * (vocabulary 4 .. 7) are 0 .. 3, every other token is the gap state 4 (q = 5).
 * rnamsm_msa_seq_weights: row k is a neighbour of row n iff (double) m(n, k) >= theta * (double) L, with m the number of
 * columns whose states are equal (gap == gap counts), 0 < theta <= 1; weights_out[n] = 1.0 / (neighbour count, itself
 * included), float64 [N]; neff_out[0] = sum_n weights_out[n], float64.  The counts are exact integers.
 * rnamsm_msa_dca: those weights, then mean-field DCA with pseudocount 0 < pseudocount < 1:
 *   f_i(a) = (1 - lam) / Neff sum_n w_n [s_ni = a] + lam / q,  f_ij(a, b) = (1 - lam) / Neff sum_n w_n [s_ni = a][s_nj = b]
 *   + lam / q^2 (i != j),  Cov[(i, a), (j, b)] = f_ij(a, b) - f_i(a) f_j(b) for a, b < 4 (f_ii(a, b) = f_i(a) d_ab),
 *   e = -Cov^-1 (blocked float64 Cholesky factorisation and inverse), F[i, j] = Frobenius norm of the 4 x 4 block e_ij
 *   padded with a zero gap row and column and put in the zero-sum gauge, F[i, i] = 0; contacts_out [L, L] fp32: the
 *   APC and symmetrisation of rnamsm_jacobian_contacts applied to F.
 * Fixed-order reductions, no atomics: bitwise reproducible.  A non-positive pivot of the factorisation leaves
 * 1 + its index in the int32 at the start of the workspace (0 otherwise; read it after the stream has run); the
 * contacts are then not valid.  Both entries enqueue only: no synchronisation, no allocation.  workspace:
 * rnamsm_seq_weights_workspace_bytes(N, L) / rnamsm_dca_workspace_bytes(N, L) bytes, 256 B aligned (0 = invalid
 * arguments); the DCA one holds two float64 matrices of side 4L rounded up to 64. */
size_t rnamsm_seq_weights_workspace_bytes(int N, int L);
int rnamsm_msa_seq_weights(const int64_t* tokens, int N, int C, double theta, double* weights_out, double* neff_out,
                           void* workspace, size_t workspace_bytes, void* stream);
size_t rnamsm_dca_workspace_bytes(int N, int L);
int rnamsm_msa_dca(const int64_t* tokens, int N, int C, double theta, double pseudocount, double* weights_out,
                   double* neff_out, float* contacts_out, void* workspace, size_t workspace_bytes, void* stream);

/* Nested secondary structure from a pair map (csrc/fold.cu; DESIGN.md 4.15; tests/fold_ref.py restates it).  maps:
 * host array of n device pointers to fp32 [L[m], L[m]] maps, of which only the upper triangle S[i, j], i < j, is read.
 * A pair (i, j) is allowed iff j - i > min_loop (>= 0), S[i, j] > threshold (finite) and, with canonical != 0,
 * {s_i, s_j} is AU, GC or GU in either order; seqs: host array of n device pointers to uint8 codes [L[m]], A G C U =
 * 0 1 2 3, any other code never pairs (may be NULL without canonical).
 *   RNAMSM_FOLD_MEA (maximum expected accuracy, S pair probabilities): w[i, j] = fp32(2 gamma) * S[i, j],
 *     u[i] = fp32(1 - sum_{j != i} S[min(i, j), max(i, j)]) summed in float64 over ascending j;  gamma > 0.
 *   RNAMSM_FOLD_SCORE (maximum-weight nested matching of any score): w[i, j] = S[i, j], u[i] = 0;  gamma ignored.
 *   P[i][k] = w[i, k] + M[i+1][k-1] for an allowed pair, else -inf;  M[i][j] = max(M[i+1][j] + u[i],
 *   max_{i < k <= j} P[i][k] + M[k+1][j]), fp32, M of an empty interval 0.  Traceback from (0, L - 1): i unpaired if
 *   M[i][j] == M[i+1][j] + u[i], else paired with the smallest k matching.  pairs_out[m]: int32 [L[m]] device, partner
 *   or -1;  scores_out: fp32 [n] device, M[0][L - 1].
 * The result is bit-identical whatever the batch.  The int32 at the start of the workspace gets bit 1 for a non-finite
 * S[i, j] (i < j) and bit 2 for a w or u that overflows fp32 (0 otherwise; read it after the stream has run); the
 * outputs are then not valid.  Launches: 1 + ceil(L_max / T) + 1, T = 32 for L_max <= 1024, else 64.  Enqueues only: no
 * synchronisation, no allocation.  workspace: rnamsm_fold_workspace_bytes(n, L) bytes (0 = invalid arguments),
 * 256 B aligned, dominated by two fp32 tables of about L x L per map. */
enum { RNAMSM_FOLD_MEA = 0, RNAMSM_FOLD_SCORE = 1 };
size_t rnamsm_fold_workspace_bytes(int n, const int* L);
int rnamsm_fold(int n, const float* const* maps, const int* L, const uint8_t* const* seqs, int mode, double gamma,
                float threshold, int min_loop, int canonical, int* const* pairs_out, float* scores_out,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- one deep MSA sharded over the GPUs of a box (SURVEY.md 8e; rna-msm_b200/sharded.py) -----------
 * The reference has no multi-GPU forward; these entry points implement the partition its math allows:
 * rows for the tied row attention (sum of partial logits over ranks), columns for the column attention
 * (it attends over rows, modules.py:907).  One process per GPU.  Buffers other GPUs touch come from
 * rnamsm_peer_alloc and are mapped into the peers through CUDA IPC handles that the host exchanges
 * (torch.distributed); the kernels below then read / write peer memory directly over NVLink.  Ordering
 * between GPUs (a phase must have finished everywhere before the next reads its results) is the
 * caller's job: a stream-ordered barrier between phases. */
int rnamsm_peer_alloc(size_t bytes, void** out);            /* cudaMalloc, zero-filled, IPC-exportable */
int rnamsm_peer_free(void* p);
int rnamsm_ipc_export(const void* p, void* handle64);       /* 64-byte cudaIpcMemHandle_t */
int rnamsm_ipc_import(const void* handle64, void** out);    /* maps a peer's buffer (enables peer access) */
int rnamsm_ipc_close(void* p);

/* LayerNorm of this rank's row shard x [Rn*C, D] (rows r0..r0+Rn of an R-row MSA) whose 16-bit output
 * rows go straight into the column owners' buffers: token (r, c) -> peer_dst[c / (C/n)], row
 * (c % (C/n)) * R + r, i.e. each peer ends with its column shard in [C/n, R, D] (column-major) order.
 * Replaces LayerNorm + the row->column all-to-all.  0 <= r0 and r0 + Rn <= R. */
int rnamsm_layernorm_push(const float* x, const float* w, const float* b, void* const* peer_dst, int n_ranks, int Rn,
                          int C, int R, int r0, int D, float eps, int y_dtype, void* stream);

/* Tied-logit exchange fused with K5: rank `rank` owns query rows [rank*C/n, (rank+1)*C/n); it pulls
 * those rows of every rank's partial logits (peer_partial[g]: fp32 [n_splits, H, C, C]), sums them,
 * applies logit_scale / key mask / softmax, writes the fp32 map rows it owns into map_out (THIS rank's
 * [H, C, C] map slab of the layer, or NULL; rows of other owners are left untouched) and the 16-bit
 * probabilities into every rank's peer_probs[g] [H, C, ld_lp] (columns >= C zero-filled).  Replaces all-reduce +
 * rnamsm_row_softmax. */
int rnamsm_row_softmax_p2p(void* const* peer_partial, int n_ranks, int rank, int n_splits, int H, int C,
                           const uint8_t* key_pad, float logit_scale, float* map_out, void* const* peer_probs,
                           int ld_lp, int dtype, void* stream);

/* Stream-ordered barrier across the ranks in peer memory (no NCCL call): peer_flags[g] is rank g's flag array
 * (>= n_ranks uint32, zero-initialised by rnamsm_peer_alloc).  `epoch` must be the same on every rank and grow by
 * one per barrier.  Work enqueued after it on `stream` starts once every rank's stream has reached its own call;
 * all peer writes of kernels enqueued before it are visible.  A peer that never arrives traps after ~10 s. */
int rnamsm_peer_barrier(void* const* peer_flags, int n_ranks, int rank, unsigned int epoch, void* stream);

/* Query rows [i0, i1) of one layer's maps (device, fp32 [H, C, C]) -> host_layer [H, Ls, Ls] with the first `start`
 * rows/columns stripped (RNA_MSM_Inference.py:150-158), one pitched DMA on `stream`.  host_layer should be pinned
 * (rnamsm_host_register) for the copy to be asynchronous. */
int rnamsm_copy_map_rows_d2h(const float* maps_layer, int H, int C, int i0, int i1, int start, int Ls, float* host_layer,
                             void* stream);

/* Page-lock / unlock a host range in this process's CUDA context (e.g. a POSIX shared-memory mapping that all
 * ranks of the box write their map rows into). */
int rnamsm_host_register(void* p, size_t bytes);
int rnamsm_host_unregister(void* p);

/* Column block's out-projection fused with the column->row exchange: ctx [R*Cn, K] (this rank's column
 * shard c0..c0+Cn, token-major (r, c_local)) x W[N, K]^T + bias[N], delivered to rank r / Rn at row
 * (r % Rn) * C + c0 + c_local of peer_x[r / Rn] ([Rn*C, N]):
 *   as_delta16 = 0: peer_x are the fp32 residual streams, the epilogue TMA-reduce-adds into them
 *                   (GEMM + exchange + residual add in one kernel; 4 bytes per element over NVLink);
 *   as_delta16 = 1: peer_x are 16-bit receive buffers, the epilogue TMA-stores the result (2 bytes per
 *                   element); the owner adds it with rnamsm_add_layernorm on its next LayerNorm pass.
 * Cn % 16 == 0.  The shard is one of the n_ranks shards of C: c0 >= 0, c0 % Cn == 0, c0 + Cn <= C, c0 / Cn < n_ranks. */
int rnamsm_linear_residual_scatter(const void* ctx, const void* W, const float* bias, int R, int Cn, int N, int K,
                                   int dtype, void* const* peer_x, int n_ranks, int Rn, int C, int c0, int as_delta16,
                                   void* stream);

/* x (fp32, in place) += delta (16-bit); y = LayerNorm(x) in 16 bits: the residual add of a contribution
 * that arrived in a receive buffer, fused into the LayerNorm that reads x next (modules.py:385-401). */
int rnamsm_add_layernorm(float* x, const void* delta, int delta_dtype, const float* w, const float* b, void* y,
                         int y_dtype, long long n_rows, int D, float eps, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RNAMSM_B200_H_ */
