// Small kernels of the LM-head scoring path (rnamsm_msa_masked_marginals in api.cu): the masked variant grids of one
// alignment, the gather of the one row each grid is scored at, and the 12-wide log-softmax over the vocabulary.
// Everything else on that path is the forward's own launches.  All three are HBM- or latency-bound.
//
// Entry k of a pass is grid k with token (row, cols[k]) masked.  An entry whose column is out of range or names a pad
// token of the row is left unmasked, gathers zeros and comes back as a row of NaN; nothing is read or written out of
// bounds for it.  The variant kernel also builds the substituted grids of the categorical Jacobian (jacobian.cu): there
// token (row, cols[k]) becomes toks[k] instead of the mask token.
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

__device__ __forceinline__ bool score_col_ok(const int64_t* __restrict__ tokens, int row, int C, int col, int pad_idx) {
  return col >= 0 && col < C && tokens[(long long)row * C + col] != pad_idx;
}

// out[k * T + t] = tokens[t], except (row, cols[k]) -> toks[k], or mask_idx when toks is NULL
__global__ void __launch_bounds__(256)
score_variants_kernel(const int64_t* __restrict__ tokens, long long T, int row, int C, const int* __restrict__ cols,
                      const int* __restrict__ toks, int n, int mask_idx, int pad_idx, int64_t* __restrict__ out) {
  const long long total = (long long)n * T;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i / T);
    const long long t = i - (long long)k * T;
    const int c = cols[k];
    const bool hit = t == (long long)row * C + c && score_col_ok(tokens, row, C, c, pad_idx);
    out[i] = hit ? (int64_t)(toks ? toks[k] : mask_idx) : tokens[t];
  }
}

// out[k, :] = x[k * grid_stride + row * C + cols[k], :] (zeros for an invalid column); one block per entry
__global__ void __launch_bounds__(128)
score_gather_kernel(const float* __restrict__ x, long long grid_stride, int row, int C, const int* __restrict__ cols,
                    int D, float* __restrict__ out) {
  const int k = blockIdx.x;
  const int c = cols[k];
  const bool ok = c >= 0 && c < C;
  const float4* src = reinterpret_cast<const float4*>(x + ((long long)k * grid_stride + (long long)row * C + (ok ? c : 0)) * D);
  float4* dst = reinterpret_cast<float4*>(out + (long long)k * D);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = ok ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
}

// One warp per entry, lane v = vocabulary entry v (V <= 32): lp holds the logits on entry and their log_softmax on exit
// (max-subtract, expf sum, logf); logits_out (optional) receives a copy of the logits.
__global__ void __launch_bounds__(256)
score_log_softmax_kernel(float* __restrict__ lp, float* __restrict__ logits_out, int n, int V,
                         const int64_t* __restrict__ tokens, int row, int C, const int* __restrict__ cols, int pad_idx) {
  const int k = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (k >= n) return;
  const bool ok = score_col_ok(tokens, row, C, cols[k], pad_idx);
  const float v = lane < V ? lp[(long long)k * V + lane] : -INFINITY;
  const float m = warp_max(v);
  const float s = warp_sum(lane < V ? expf(v - m) : 0.f);
  const float ls = logf(s);
  if (lane < V) {
    if (logits_out) logits_out[(long long)k * V + lane] = ok ? v : NAN;
    lp[(long long)k * V + lane] = ok ? (v - m) - ls : NAN;
  }
}

int launch_score_variants(const int64_t* tokens, long long T, int row, int C, const int* cols, const int* toks, int n,
                          int mask_idx, int pad_idx, int64_t* out, cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && T > 0, "score_variants: empty pass (n=%d T=%lld)", n, T);
  const long long total = (long long)n * T;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 148LL * 16);
  score_variants_kernel<<<blocks, 256, 0, st>>>(tokens, T, row, C, cols, toks, n, mask_idx, pad_idx, out);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_score_gather(const float* x, long long grid_stride, int row, int C, const int* cols, int n, int D, float* out,
                        cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && D % 4 == 0, "score_gather: n=%d D=%d", n, D);
  score_gather_kernel<<<n, 128, 0, st>>>(x, grid_stride, row, C, cols, D, out);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_score_log_softmax(float* lp, float* logits_out, int n, int V, const int64_t* tokens, int row, int C,
                             const int* cols, int pad_idx, cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && V >= 1 && V <= 32, "score_log_softmax: n=%d V=%d (V <= 32)", n, V);
  score_log_softmax_kernel<<<ceil_div(n, 8), 256, 0, st>>>(lp, logits_out, n, V, tokens, row, C, cols, pad_idx);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rnamsm
