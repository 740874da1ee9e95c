// Kernels of iterative masked sampling with the LM head (rnamsm_msa_gibbs_sample in api.cu): the mask draw over the
// chains' states, the gather of the sampled rows' pre-final-LayerNorm states, and the draw of each masked token from
// its logits.  Everything else on that path is the forward's own launches.  All three are HBM- or latency-bound.
//
// Random numbers: Philox4x32-10 (Salmon et al., SC'11; the Random123 reference), stateless, so a draw depends only on
// its coordinates and never on how chains are grouped into passes or steps into calls.
//   key     = (seed & 0xffffffff, seed >> 32)
//   counter = (k, s, r * C + c, purpose)      k: chain, s: absolute step, (r, c): token, purpose 0 = mask, 1 = draw
//   u       = (word0 >> 8) * 2^-24             a uniform in [0, 1), exact in fp32 and float64 alike
// Token (r, c) of chain k is masked at step s when r is a sampled row, c >= 1, the token is not <pad> and
// u(purpose 0) < p.  A masked token is drawn from the allowed tokens' logits over T by inverse CDF with u(purpose 1):
// the smallest allowed v (in index order) with u * S < W_v, W_v the running sum of exp((l_v - max) / T) and S the total
// (the last allowed v if rounding leaves none); T = 0 takes the argmax, ties to the lowest index.
//
// Entry (i, j, c) of a pass is chain k0 + i, sampled row rows[j], column c.  A row out of [0, R) is never masked,
// gathers zeros and draws nothing.
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t lo0 = 0xD2511F53u * ctr.x, hi0 = __umulhi(0xD2511F53u, ctr.x);
    const uint32_t lo1 = 0xCD9E8D57u * ctr.z, hi1 = __umulhi(0xCD9E8D57u, ctr.z);
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

__device__ __forceinline__ float sample_uniform(unsigned long long seed, int k, int s, long long t, uint32_t purpose) {
  const uint4 w = philox4x32_10(make_uint4((uint32_t)k, (uint32_t)s, (uint32_t)t, purpose),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  return (float)(w.x >> 8) * 0x1p-24f;
}

struct SampleStep {
  unsigned long long seed;
  int k0, step, R, C, n_rows, pad_idx;
  long long T;
  float p;
};

// whether token (r, c) of chain k (state: its [R, C] tokens) is masked at this step
__device__ __forceinline__ bool sample_masked(const SampleStep& a, const int64_t* __restrict__ state, int k, int r, int c) {
  if (r < 0 || r >= a.R || c < 1) return false;
  const long long t = (long long)r * a.C + c;
  return state[t] != a.pad_idx && sample_uniform(a.seed, k, a.step, t, 0u) < a.p;
}

// grids [n, T]: a copy of the pass's chain states on entry; mask_idx at this step's masked tokens on exit
__global__ void __launch_bounds__(256)
sample_mask_kernel(SampleStep a, const int64_t* __restrict__ states, const int* __restrict__ rows, int n, int mask_idx,
                   int64_t* __restrict__ grids) {
  const long long per = (long long)a.n_rows * a.C, total = (long long)n * per;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / per);
    const int j = (int)((e - i * per) / a.C);
    const int c = (int)(e - i * per - (long long)j * a.C);
    const int r = rows[j];
    if (sample_masked(a, states + (long long)(a.k0 + i) * a.T, a.k0 + i, r, c))
      grids[i * a.T + (long long)r * a.C + c] = mask_idx;
  }
}

// out[(i * n_rows + j) * C + c, :] = x[i * T + rows[j] * C + c, :]; one block per (i, j), zeros for a row out of range
__global__ void __launch_bounds__(256)
sample_gather_rows_kernel(const float* __restrict__ x, long long T, int R, int C, const int* __restrict__ rows, int n_rows,
                          int D, float* __restrict__ out) {
  const int i = blockIdx.x / n_rows, j = blockIdx.x - i * n_rows;
  const int r = rows[j];
  const bool ok = r >= 0 && r < R;
  const long long n4 = (long long)C * D / 4;
  const float4* src = reinterpret_cast<const float4*>(x + ((long long)i * T + (long long)(ok ? r : 0) * C) * D);
  float4* dst = reinterpret_cast<float4*>(out + (long long)blockIdx.x * C * D);
  for (long long q = threadIdx.x; q < n4; q += blockDim.x) dst[q] = ok ? src[q] : make_float4(0.f, 0.f, 0.f, 0.f);
}

// One warp per entry, lane v = vocabulary entry v (V <= 32).  logits [n * n_rows * C, V]; the draw goes into the
// chain's state.  Entries that are not masked leave the state alone.
__global__ void __launch_bounds__(256)
sample_draw_kernel(SampleStep a, const float* __restrict__ logits, int V, float temperature, uint32_t allowed, int n,
                   const int* __restrict__ rows, int64_t* __restrict__ states) {
  const long long e = (long long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  const long long per = (long long)a.n_rows * a.C;
  if (e >= (long long)n * per) return;
  const int i = (int)(e / per);
  const int j = (int)((e - i * per) / a.C);
  const int c = (int)(e - i * per - (long long)j * a.C);
  const int r = rows[j];
  const int k = a.k0 + i;
  int64_t* state = states + (long long)k * a.T;
  if (!sample_masked(a, state, k, r, c)) return;   // warp-uniform
  const bool ok = lane < V && ((allowed >> lane) & 1u);
  const float l = ok ? logits[e * V + lane] : -INFINITY;
  const float m = warp_max(l);
  unsigned hit;
  if (temperature == 0.f) {
    hit = __ballot_sync(0xffffffffu, ok && l == m);
  } else {
    float W = ok ? expf((l - m) / temperature) : 0.f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float y = __shfl_up_sync(0xffffffffu, W, o);
      if (lane >= o) W += y;
    }
    const float S = __shfl_sync(0xffffffffu, W, 31);
    const float u = sample_uniform(a.seed, k, a.step, (long long)r * a.C + c, 1u);
    hit = __ballot_sync(0xffffffffu, ok && u * S < W);
  }
  const int v = hit ? __ffs(hit) - 1 : 31 - __clz(allowed);
  if (lane == 0) state[(long long)r * a.C + c] = v;
}

static SampleStep sample_step(unsigned long long seed, int k0, int step, int R, int C, int n_rows, int pad_idx, float p) {
  return SampleStep{seed, k0, step, R, C, n_rows, pad_idx, (long long)R * C, p};
}

int launch_sample_mask(const int64_t* states, int64_t* grids, int n, int R, int C, const int* rows, int n_rows, int pad_idx,
                       int mask_idx, float p, unsigned long long seed, int k0, int step, cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && n_rows > 0 && R > 0 && C > 0, "sample_mask: empty pass (n=%d n_rows=%d R=%d C=%d)", n, n_rows, R, C);
  const SampleStep a = sample_step(seed, k0, step, R, C, n_rows, pad_idx, p);
  const long long total = (long long)n * n_rows * C;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 148LL * 16);
  sample_mask_kernel<<<blocks, 256, 0, st>>>(a, states, rows, n, mask_idx, grids);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_sample_gather_rows(const float* x, int n, int R, int C, const int* rows, int n_rows, int D, float* out,
                              cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && n_rows > 0 && D % 4 == 0 && (long long)n * n_rows < (1LL << 31),
                 "sample_gather_rows: n=%d n_rows=%d D=%d", n, n_rows, D);
  sample_gather_rows_kernel<<<n * n_rows, 256, 0, st>>>(x, (long long)R * C, R, C, rows, n_rows, D, out);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_sample_draw(const float* logits, int V, float temperature, unsigned allowed, int64_t* states, int n, int R, int C,
                       const int* rows, int n_rows, int pad_idx, float p, unsigned long long seed, int k0, int step,
                       cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && n_rows > 0 && V >= 1 && V <= 32 && allowed != 0 && (V == 32 || (allowed >> V) == 0),
                 "sample_draw: n=%d n_rows=%d V=%d allowed=0x%x (V <= 32, allowed a non-empty subset of the vocabulary)",
                 n, n_rows, V, allowed);
  const SampleStep a = sample_step(seed, k0, step, R, C, n_rows, pad_idx, p);
  const long long warps = (long long)n * n_rows * C;
  const long long blocks = (warps + 7) / 8;
  RNAMSM_REQUIRE(blocks < (1LL << 31), "sample_draw: %lld entries", warps);
  sample_draw_kernel<<<(unsigned)blocks, 256, 0, st>>>(a, logits, V, temperature, allowed, n, rows, states);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rnamsm
