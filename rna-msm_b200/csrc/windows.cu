// Full-length features for sequences longer than the learned column positions: the window plan, the kernel that builds
// a pass of window grids, and the stitch kernel of rnamsm_msa_forward_windows (api.cu).
//
// Input [R, C] with BOS at column 0 and L = C - 1 residues.  W = min(window, L); window k (0-based) starts at residue
//   s_k = min(k * stride, L - W),  k < K = 1 + ceil((L - W) / stride)
// and its grid is [R, W + 1]: column 0 of the input, then input columns 1 + s_k .. W + s_k.  Each window runs as an MSA
// of its own (positions restart), giving emb_k [W, D] (row 0 of the final representation, BOS stripped), the N*H maps
// map_k [N*H, W, W] and optionally the contacts [W, W].
//
// Stitching (tests/windows_ref.py restates it in float64 numpy).  Tent weight of residue p in window k:
//   w_k(p) = min(p - s_k + 1, s_k + W - p)       (an integer >= 1 inside the window)
//   emb[p]       = sum_k c_k(p) emb_k[p - s_k],                 c_k(p)    = w_k(p) / sum_k' w_k'(p)
//   atp[h, i, j] = sum_k c_k(i, j) map_k[h, i - s_k, j - s_k],  c_k(i, j) = w_k(i) w_k(j) / sum_k' w_k'(i) w_k'(j)
// over the windows that contain the residue (both residues); contacts use the pair weights.  A pair no window contains is
// exactly 0.  Each coefficient is the float64 quotient of the integer sums, rounded once to fp32; the sum is accumulated
// in fp32 as acc = fmaf(c_k, v_k, acc) from acc = 0 in ascending k.  Between passes the running sum lives in the fp32
// output, so the result does not depend on how the windows are grouped into passes, and an entry covered by one window
// is that window's value bit for bit (c = 1).
#include <climits>

#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

// grids [n, R, W + 1] of windows k0 .. k0 + n - 1 from tokens [R, C]
__global__ void __launch_bounds__(256)
window_build_kernel(const int64_t* __restrict__ tokens, int R, int C, const int* __restrict__ starts, int k0, int n, int W,
                    int64_t* __restrict__ grids) {
  const int Cw = W + 1;
  const long long total = (long long)n * R * Cw;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(e % Cw);
    const long long rk = e / Cw;
    const int r = (int)(rk % R), k = (int)(rk / R);
    grids[e] = tokens[(long long)r * C + (c == 0 ? 0 : c + starts[k0 + k])];
  }
}

__device__ __forceinline__ int tent(int p, int s, int W) { return min(p - s + 1, s + W - p); }

// first k in [0, K] with starts[k] >= t (starts strictly ascending)
__device__ __forceinline__ int first_start_at_least(const int* __restrict__ starts, int K, int t) {
  int lo = 0, hi = K;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (starts[mid] < t) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

constexpr int kStitchPlanes = 8;   // output planes one thread accumulates at a time

// One launch per pass of windows k0 .. k0 + n - 1.  Blocks [0, map_blocks): 32 x 8 tiles of the [L, L] pair grid, one
// pair per thread, over every plane (the N*H maps, then the contacts when cw is not NULL).  Blocks past those: one
// residue of emb each.  Output-stationary: each output element is owned by one thread, which reads the window values
// of this pass (each once) and its own running sum, so no atomics are needed.  The first pass (k0 == 0) also writes
// the zeros of the pairs that no window contains.
//   maps [n, NH, W + 1, W + 1] (BOS row / column included), cw [n, W, W], hx [n, W + 1, D]
__global__ void __launch_bounds__(256)
window_stitch_kernel(const float* __restrict__ maps, int NH, const float* __restrict__ cw, const float* __restrict__ hx,
                     int D, const int* __restrict__ starts, int K, int k0, int n, int W, int L, int tiles_j,
                     int map_blocks, float* __restrict__ emb_out, float* __restrict__ atp_out,
                     float* __restrict__ contacts_out) {
  const int Cw = W + 1;
  const int kl = k0 + n - 1;   // last window of the pass
  if ((int)blockIdx.x >= map_blocks) {
    const int p = (int)blockIdx.x - map_blocks;
    const int ka = first_start_at_least(starts, K, p - W + 1), kb = first_start_at_least(starts, K, p + 1) - 1;
    const int qa = max(ka, k0), qb = min(kb, kl);
    if (qa > qb) return;
    long long den = 0;
    for (int k = ka; k <= kb; ++k) den += tent(p, starts[k], W);
    const bool first = ka >= k0;
    for (int d = threadIdx.y * blockDim.x + threadIdx.x; d < D; d += blockDim.x * blockDim.y) {
      float acc = first ? 0.f : emb_out[(size_t)p * D + d];
      for (int k = qa; k <= qb; ++k) {
        const int s = starts[k];
        const float c = (float)((double)tent(p, s, W) / (double)den);
        acc = fmaf(c, hx[((size_t)(k - k0) * Cw + p - s + 1) * D + d], acc);
      }
      emb_out[(size_t)p * D + d] = acc;
    }
    return;
  }
  const int i = ((int)blockIdx.x / tiles_j) * 8 + threadIdx.y;
  const int j = ((int)blockIdx.x % tiles_j) * 32 + threadIdx.x;
  if (i >= L || j >= L) return;
  const int n_planes = NH + (cw ? 1 : 0);
  const size_t LL = (size_t)L * L, o = (size_t)i * L + j;
  auto plane = [&](int q) -> float* { return q < NH ? atp_out + (size_t)q * LL : contacts_out; };
  const int lo = min(i, j), hi = max(i, j);
  const int ka = first_start_at_least(starts, K, hi - W + 1), kb = first_start_at_least(starts, K, lo + 1) - 1;
  if (ka > kb) {   // no window contains the pair
    if (k0 == 0)
      for (int q = 0; q < n_planes; ++q) plane(q)[o] = 0.f;
    return;
  }
  const int qa = max(ka, k0), qb = min(kb, kl);
  if (qa > qb) return;
  long long den = 0;
  for (int k = ka; k <= kb; ++k) den += (long long)tent(i, starts[k], W) * tent(j, starts[k], W);
  const double dden = (double)den;
  const bool first = ka >= k0;
  const size_t map_sz = (size_t)Cw * Cw;
  for (int q0 = 0; q0 < n_planes; q0 += kStitchPlanes) {
    float acc[kStitchPlanes];
#pragma unroll
    for (int u = 0; u < kStitchPlanes; ++u) acc[u] = (first || q0 + u >= n_planes) ? 0.f : plane(q0 + u)[o];
    for (int k = qa; k <= qb; ++k) {
      const int s = starts[k];
      const float c = (float)((double)((long long)tent(i, s, W) * tent(j, s, W)) / dden);
      const int a = i - s, b = j - s;
      const float* mk = maps + (size_t)(k - k0) * NH * map_sz + (size_t)(a + 1) * Cw + b + 1;
#pragma unroll
      for (int u = 0; u < kStitchPlanes; ++u) {
        const int q = q0 + u;
        if (q < NH) acc[u] = fmaf(c, mk[(size_t)q * map_sz], acc[u]);
        else if (q < n_planes) acc[u] = fmaf(c, cw[((size_t)(k - k0) * W + a) * W + b], acc[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < kStitchPlanes; ++u)
      if (q0 + u < n_planes) plane(q0 + u)[o] = acc[u];
  }
}

// -> K, writing the starts when starts_out is not NULL; 0 (with the reason in rnamsm_last_error) for invalid arguments
int window_starts(int L, int window, int stride, int* starts_out) {
  if (L < 1) {
    set_error("window_starts: L=%d (need at least one residue)", L);
    return 0;
  }
  if (stride < 1 || stride > window) {
    set_error("window_starts: need 1 <= stride <= window (stride=%d window=%d)", stride, window);
    return 0;
  }
  const int W = std::min(window, L);
  const int K = (int)(1 + ((long long)L - W + stride - 1) / stride);
  if (starts_out)
    for (int k = 0; k < K; ++k) starts_out[k] = (int)std::min<long long>((long long)k * stride, L - W);
  return K;
}

int launch_window_build(const int64_t* tokens, int R, int C, const int* starts, int k0, int n, int W, int64_t* grids,
                        cudaStream_t st) {
  const long long total = (long long)n * R * (W + 1);
  RNAMSM_REQUIRE(total > 0, "window_build: empty pass (n=%d R=%d W=%d)", n, R, W);
  ProfScope prof(KC_WINDOW_BUILD, st);
  window_build_kernel<<<(int)std::min<long long>((total + 255) / 256, 148LL * 16), 256, 0, st>>>(tokens, R, C, starts, k0,
                                                                                                 n, W, grids);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_window_stitch(const float* maps, int NH, const float* cw, const float* hx, int D, const int* starts, int K,
                         int k0, int n, int W, int L, float* emb_out, float* atp_out, float* contacts_out, cudaStream_t st) {
  RNAMSM_REQUIRE(n >= 1 && k0 >= 0 && k0 + n <= K && W >= 1 && L >= W && NH >= 1 && D >= 1,
                 "window_stitch: bad pass (k0=%d n=%d K=%d W=%d L=%d)", k0, n, K, W, L);
  const int tiles_j = ceil_div(L, 32);
  const long long map_blocks = (long long)ceil_div(L, 8) * tiles_j;
  RNAMSM_REQUIRE(map_blocks + L <= INT_MAX, "window_stitch: L=%d too large", L);
  ProfScope prof(KC_WINDOW_STITCH, st);
  window_stitch_kernel<<<(int)(map_blocks + L), dim3(32, 8), 0, st>>>(maps, NH, cw, hx, D, starts, K, k0, n, W, L, tiles_j,
                                                                    (int)map_blocks, emb_out, atp_out, contacts_out);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" int rnamsm_window_starts(int L, int window, int stride, int* starts_out) {
  return window_starts(L, window, stride, starts_out);
}
