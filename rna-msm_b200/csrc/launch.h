// Internal launcher declarations shared by the translation units of librnamsm_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

namespace rnamsm {

void count_launch(int n = 1);
long long launch_count();

// Optional per-kernel-class device timing (cudaEvents on the launching stream), used by bench.py
// for the live roofline figure and the per-kernel time shares.  Off by default: zero overhead.
enum KernelClass {
  KC_EMBED_LN = 0, KC_LAYERNORM, KC_ROW_SOFTMAX, KC_VOCAB_PROJ, KC_LINEAR_QKV, KC_LINEAR_FC1, KC_LINEAR_OUT,
  KC_LINEAR_FC2, KC_ROW_LOGITS, KC_ROW_AV, KC_COL_ATTN, KC_CONTACT, KC_ROW_SHORT, KC_WINDOW_BUILD,
  KC_WINDOW_STITCH, KC_COUNT
};
struct ProfScope {
  int cls;
  cudaStream_t st;
  void* slot;
  ProfScope(int cls, cudaStream_t st);
  ~ProfScope();
};

// elementwise.cu
int launch_embed_ln(const int64_t* tokens, int R, int C, const float* tok_emb, int vocab, const float* pos_emb,
                    int n_pos, const float* row_pos, const float* ln_w, const float* ln_b, int D, int pad_idx,
                    float eps, float* x_out, uint8_t* pad_out, cudaStream_t st);
// tr_R, tr_C > 0: write the output in column-major token order, y[c * tr_R + r] = LN(x[r * tr_C + c])
// x_dtype != 0: x holds 16-bit rows (1 = bf16, 2 = fp16; fp32 output only)
int launch_layernorm(const float* x, const float* w, const float* b, void* y, int y_dtype, long long n_rows, int D,
                     float eps, cudaStream_t st, int tr_R = 0, int tr_C = 0, int x_dtype = 0);
int launch_row_softmax(const float* partial, int n_splits, int H, int C, const uint8_t* key_pad, float logit_scale,
                       float* probs_out, void* probs_lp, int ld_lp, int dtype, cudaStream_t st);
int launch_vocab_proj(const float* h, const float* E, const float* bias, long long M, int V, int D, float* out,
                      cudaStream_t st);

// debug: count 16-bit elements at / beyond the largest finite value, track max |v| (counters: 2 x u64 on the device)
int launch_range_scan(const void* p, long long n, int dtype, unsigned long long* counters, cudaStream_t st);

// Epilogue description shared by the fp32 (FFMA) and 16-bit (tcgen05) linear kernels.
struct LinearEpilogue {
  int kind;                 // RNAMSM_EPI_*
  const float* bias;        // [N]
  float q_scale;            // applied to columns [0, q_cols) after the bias
  int q_cols;
  const uint8_t* row_mask;  // [M] or nullptr; zeroes columns [0, q_cols) of masked rows
};

// Kernel class of a dense linear launch (for the timing breakdown): by epilogue and shape.
inline int linear_class(int epi_kind, int N, int K) {
  if (epi_kind == 1) return KC_LINEAR_FC1;
  if (epi_kind == 2) return K > N ? KC_LINEAR_FC2 : KC_LINEAR_OUT;
  return KC_LINEAR_QKV;
}

// simt_f32.cu -- fp32 parity path
int launch_linear_f32(const float* x, const float* W, long long M, int N, int K, const LinearEpilogue& epi, float* out,
                      cudaStream_t st);
int launch_row_logits_f32(const float* qkv, int R, int C, int H, float* partial, int n_splits, cudaStream_t st);
int launch_row_av_f32(const float* probs, int ldp, const float* qkv, int R, int C, int H, float* ctx, cudaStream_t st);
int launch_col_attn_f32(const float* qkv, int R, int C, int H, const uint8_t* pad, float* ctx, cudaStream_t st);

// LayerNorm fused behind a residual epilogue: y = LN(out) (full rows of N features, fp32 statistics), 16-bit.
struct LnFuse {
  const float* w;
  const float* b;
  float eps;
  void* out;          // [M, N] 16-bit
  int out_fp16;       // 0 = bf16, 1 = fp16
  int tr_R, tr_C;     // > 0: output row (m % tr_C) * tr_R + m / tr_C
  int* counters;      // >= 2 * ceil(M / 256) ints, ZERO on entry (the kernel leaves them zero again)
};
inline size_t ln_counter_bytes(long long M) { return (size_t)(2 * ((M + 255) / 256)) * sizeof(int); }

// umma_gemm.cu -- 16-bit (bf16 / fp16 operands, fp32 accumulate) tcgen05 path; fp16 != 0 selects fp16
int launch_linear_16(const void* x, const void* W, long long M, int N, int K, int fp16, const LinearEpilogue& epi,
                     void* out, cudaStream_t st, const LnFuse* ln = nullptr);
// fp32 linear on the tensor cores: hi / lo tf32 split of both operands, three kind::tf32 MMAs per k-step
int launch_linear_tf32(const float* x_hi, const float* x_lo, const float* W_hi, const float* W_lo, long long M, int N, int K,
                       const LinearEpilogue& epi, float* out, cudaStream_t st);
// hi = x with the low 13 mantissa bits cleared (a tf32 number), lo = x - hi (exact); n elements
int launch_split_tf32(const float* x, float* hi, float* lo, long long n, cudaStream_t st);
int launch_row_logits_16(const void* qkv, int R, int C, int H, int fp16, float* partial, int n_splits, cudaStream_t st);
int launch_row_av_16(const void* probs, int ldp, const void* qkv, int R, int C, int H, int fp16, void* ctx,
                     cudaStream_t st);
int row_logits_splits_16(int R, int C, int H);
int gemm_max_pairs();
int launch_linear_16_scatter(const void* x, const void* W, const float* bias, int R, int Cn, int N, int K, int fp16,
                             void* const* peer_x, int n_ranks, int Rn, int C, int c0, int as_delta16, cudaStream_t st);
int launch_add_layernorm(float* x, const void* delta, int delta_dtype, const float* w, const float* b, void* y,
                         int y_dtype, long long n_rows, int D, float eps, cudaStream_t st);

// row_attn_short.cu -- the whole tied row attention of a short alignment (C <= 128) in one cooperative launch:
// partial logits per (head, row chunk) -> grid barrier -> softmax (fp32 map + 16-bit P) -> grid barrier -> P V.
// row_attn_short_chunks: the chunk (= split) count that path uses for a shape, 0 when it does not apply.
int row_attn_short_chunks(int R, int C, int H);
int launch_row_attn_short_16(const void* qkv, int R, int C, int H, int fp16, float* partial, int n_chunks, const uint8_t* key_pad,
                             float logit_scale, float* map, void* probs_lp, int ldp, void* ctx, cudaStream_t st);

// col_attn_umma.cu
int launch_col_attn_16(const void* qkv, int R, int C, int H, int fp16, int col_major, const uint8_t* pad, void* ctx,
                       cudaStream_t st);

// col_attn_probs.cu -- column-attention probabilities P [H, C, R, R] and / or their column mean [H, R, R] (either may
// be NULL); dtype RNAMSM_F32 / BF16 / F16; scratch: col_probs_scratch_bytes(R, C, H) bytes (per-row max and log-sum)
size_t col_probs_scratch_bytes(int R, int C, int H);
int launch_col_probs(const void* qkv, int R, int C, int H, int dtype, int col_major, const uint8_t* pad, float* probs,
                     float* mean, void* scratch, cudaStream_t st);

// score.cu -- LM-head scoring: n variant grids of T tokens with (row, cols[k]) masked (set to toks[k] when toks is not
// NULL: the substituted grids of the categorical Jacobian); the pre-final-LayerNorm row
// (row, cols[k]) of grid k (grids grid_stride tokens apart) into out [n, D]; log_softmax of lp [n, V] in place, with
// the logits copied to logits_out (optional).  Invalid columns (out of range, pad) give NaN rows.
int launch_score_variants(const int64_t* tokens, long long T, int row, int C, const int* cols, const int* toks, int n,
                          int mask_idx, int pad_idx, int64_t* out, cudaStream_t st);
int launch_score_gather(const float* x, long long grid_stride, int row, int C, const int* cols, int n, int D, float* out,
                        cudaStream_t st);
int launch_score_log_softmax(float* lp, float* logits_out, int n, int V, const int64_t* tokens, int row, int C,
                             const int* cols, int pad_idx, cudaStream_t st);

// sample.cu -- iterative masked sampling: a pass of n chains (k0 .. k0 + n - 1, states [n_chains, R, C]) over the
// sampled rows rows[0 .. n_rows).  mask: grids [n, R, C] (a copy of the pass's states) get mask_idx at this step's
// masked tokens; gather_rows: the sampled rows of x [n, R, C, D] into out [n, n_rows, C, D]; draw: each masked token
// drawn from logits [n, n_rows, C, V] into its chain's state.
int launch_sample_mask(const int64_t* states, int64_t* grids, int n, int R, int C, const int* rows, int n_rows, int pad_idx,
                       int mask_idx, float p, unsigned long long seed, int k0, int step, cudaStream_t st);
int launch_sample_gather_rows(const float* x, int n, int R, int C, const int* rows, int n_rows, int D, float* out,
                              cudaStream_t st);
int launch_sample_draw(const float* logits, int V, float temperature, unsigned allowed, int64_t* states, int n, int R, int C,
                       const int* rows, int n_rows, int pad_idx, float p, unsigned long long seed, int k0, int step,
                       cudaStream_t st);

// jacobian.cu -- categorical Jacobian: J[slabs[k], j, b] = logits[k * C + positions[j], alphabet[b]] -
// wt[positions[j], alphabet[b]] for the n grids of a pass (logits [n * C, V], wt [C, V]; J [P, A, P, A]).
int launch_jacobian_collect(const float* logits, const float* wt, int n, int C, int V, const int* positions, int P,
                            const int* alphabet, int A, const int* slabs, float* J, cudaStream_t st);
// contacts_out [P, P] fp32 from F [P, P] float64 with a zero diagonal: F - rowsum (x) colsum / total (0 when total == 0),
// diagonal zeroed again, then (F + F^T) / 2; sums: 2P + 1 float64 of scratch.  Shared by the Jacobian and DCA contacts.
int launch_apc_contacts(const double* F, int P, double* sums, float* out, cudaStream_t st);

// windows.cu -- overlapping windows of a long alignment: the plan (K starts, or 0 with the reason set), the grids
// [n, R, W + 1] of windows k0 .. k0 + n - 1, and the stitch of their outputs into emb [L, D], atp [NH, L, L] and
// contacts [L, L] (maps [n, NH, W + 1, W + 1], cw [n, W, W] or NULL, hx [n, W + 1, D]).
int window_starts(int L, int window, int stride, int* starts_out);
int launch_window_build(const int64_t* tokens, int R, int C, const int* starts, int k0, int n, int W, int64_t* grids,
                        cudaStream_t st);
int launch_window_stitch(const float* maps, int NH, const float* cw, const float* hx, int D, const int* starts, int K,
                         int k0, int n, int W, int L, float* emb_out, float* atp_out, float* contacts_out, cudaStream_t st);

}  // namespace rnamsm
