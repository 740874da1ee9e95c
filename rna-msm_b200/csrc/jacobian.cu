// Categorical Jacobian of the LM head (Zhang et al., PNAS 2024) for one query row: the collect kernel of
// rnamsm_msa_categorical_jacobian (api.cu), and rnamsm_jacobian_contacts, which turns J into a contact map.
//
//   J[i, a, j, b] = f(G(i, a))[j, b] - f(tokens)[j, b]        [P, A, P, A] fp32
// G(i, a): the grid with token (row, positions[i]) replaced by alphabet[a]; f(G)[j, b]: the LM-head logit of G at
// (row, positions[j]) for token alphabet[b].
//
// Contacts [P, P] from J (tests/jacobian_ref.py restates this in float64 numpy):
//   1. centre J: subtract its mean over axis i, then over a, then j, then b
//   2. F[i, j] = sqrt(sum_{a,b} J~[i, a, j, b]^2), F[i, i] = 0
//   3. average product correction as the reference's apc (utils/tensor.py:103-113): F - rowsum (x) colsum / total (term
//      0 when total == 0), diagonal zeroed again
//   4. symmetrise: (F + F^T) / 2
// Every reduction is one thread's loop in a fixed order, in float64 (no atomics), so the map is bitwise reproducible.
// These kernels are cheap next to the forwards that produce J (3P + 1 of them), so they favour plainness over speed.
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

static int grid_blocks(long long total) { return (int)std::min<long long>((total + 255) / 256, 148LL * 16); }

// J[slabs[k] * P * A + j * A + b] = logits[(k * C + positions[j]) * V + alphabet[b]] - wt[positions[j] * V + alphabet[b]]
__global__ void __launch_bounds__(256)
jacobian_collect_kernel(const float* __restrict__ logits, const float* __restrict__ wt, int n, int C, int V,
                        const int* __restrict__ positions, int P, const int* __restrict__ alphabet, int A,
                        const int* __restrict__ slabs, float* __restrict__ J) {
  const long long PA = (long long)P * A, total = (long long)n * PA;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(e / PA);
    const long long r = e - k * PA;
    const int j = (int)(r / A), b = (int)(r - (long long)j * A);
    const long long src = (long long)positions[j] * V + alphabet[b];
    J[(long long)slabs[k] * PA + r] = logits[(long long)k * C * V + src] - wt[src];
  }
}

// x viewed as [outer, n, inner]: dst = src - its mean over the middle axis.  One thread per (outer, inner) line, which
// it reads whole before it writes, so src == dst is fine.
template <typename T>
__global__ void __launch_bounds__(256)
jacobian_center_kernel(const T* src, double* dst, long long outer, int n, long long inner) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < outer * inner;
       e += (long long)gridDim.x * blockDim.x) {
    const long long o = e / inner;
    const long long base = o * n * inner + (e - o * inner);
    double s = 0.0;
    for (int q = 0; q < n; ++q) s += (double)src[base + q * inner];
    const double mean = s / n;
    for (int q = 0; q < n; ++q) dst[base + q * inner] = (double)src[base + q * inner] - mean;
  }
}

// F[i, j] = sqrt(sum_{a,b} Jc[i, a, j, b]^2), 0 on the diagonal
__global__ void __launch_bounds__(256)
jacobian_frobenius_kernel(const double* __restrict__ Jc, int P, int A, double* __restrict__ F) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)P * P;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / P), j = (int)(e - (long long)i * P);
    double s = 0.0;
    for (int a = 0; a < A; ++a)
      for (int b = 0; b < A; ++b) {
        const double v = Jc[(((long long)i * A + a) * P + j) * A + b];
        s += v * v;
      }
    F[e] = i == j ? 0.0 : sqrt(s);
  }
}

// sums[0, P): row sums of F; sums[P, 2P): column sums
__global__ void __launch_bounds__(256)
jacobian_margins_kernel(const double* __restrict__ F, int P, double* __restrict__ sums) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * P) return;
  const bool row = t < P;
  const int i = row ? t : t - P;
  double s = 0.0;
  for (int q = 0; q < P; ++q) s += F[row ? (long long)i * P + q : (long long)q * P + i];
  sums[t] = s;
}

// sums[2P] = the total of F (the row sums added in order); one thread
__global__ void jacobian_total_kernel(double* sums, int P) {
  double s = 0.0;
  for (int i = 0; i < P; ++i) s += sums[i];
  sums[2 * P] = s;
}

__device__ __forceinline__ double jacobian_apc(const double* __restrict__ F, const double* __restrict__ sums, int P, int i,
                                               int j) {
  if (i == j) return 0.0;
  const double total = sums[2 * P];
  return F[(long long)i * P + j] - (total != 0.0 ? sums[i] * sums[P + j] / total : 0.0);
}

// out[i, j] = (G[i, j] + G[j, i]) / 2, G = F - rowsum (x) colsum / total with a zero diagonal
__global__ void __launch_bounds__(256)
jacobian_contacts_kernel(const double* __restrict__ F, const double* __restrict__ sums, int P, float* __restrict__ out) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)P * P;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / P), j = (int)(e - (long long)i * P);
    out[e] = (float)(0.5 * (jacobian_apc(F, sums, P, i, j) + jacobian_apc(F, sums, P, j, i)));
  }
}

int launch_jacobian_collect(const float* logits, const float* wt, int n, int C, int V, const int* positions, int P,
                            const int* alphabet, int A, const int* slabs, float* J, cudaStream_t st) {
  RNAMSM_REQUIRE(n > 0 && C > 0 && P > 0 && A > 0, "jacobian_collect: empty pass (n=%d C=%d P=%d A=%d)", n, C, P, A);
  jacobian_collect_kernel<<<grid_blocks((long long)n * P * A), 256, 0, st>>>(logits, wt, n, C, V, positions, P, alphabet,
                                                                             A, slabs, J);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_apc_contacts(const double* F, int P, double* sums, float* out, cudaStream_t st) {
  jacobian_margins_kernel<<<ceil_div(2 * P, 256), 256, 0, st>>>(F, P, sums);
  jacobian_total_kernel<<<1, 1, 0, st>>>(sums, P);
  jacobian_contacts_kernel<<<grid_blocks((long long)P * P), 256, 0, st>>>(F, sums, P, out);
  count_launch(3);
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// scratch: Jc [P, A, P, A] float64 | F [P, P] float64 | sums [2P + 1] float64 (every region 256 B aligned)
static size_t align256_(size_t x) { return (x + 255) & ~(size_t)255; }

size_t jacobian_contacts_scratch_bytes(int P, int A) {
  const size_t PA = (size_t)P * A;
  return align256_(PA * PA * 8) + align256_((size_t)P * P * 8) + align256_((2 * (size_t)P + 1) * 8);
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

size_t rnamsm_jacobian_contacts_scratch_bytes(int P, int A) {
  if (P < 1 || A < 1) {
    set_error("jacobian_contacts: empty Jacobian (P=%d A=%d)", P, A);
    return 0;
  }
  return jacobian_contacts_scratch_bytes(P, A);
}

int rnamsm_jacobian_contacts(const float* J, int P, int A, float* contacts_out, void* scratch, size_t scratch_bytes,
                             void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  RNAMSM_REQUIRE(P >= 1 && A >= 1, "jacobian_contacts: empty Jacobian (P=%d A=%d)", P, A);
  RNAMSM_REQUIRE(J && contacts_out && scratch, "jacobian_contacts: J, contacts_out and scratch required");
  const size_t need = jacobian_contacts_scratch_bytes(P, A);
  RNAMSM_REQUIRE(scratch_bytes >= need, "jacobian_contacts: scratch %zu < required %zu", scratch_bytes, need);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "jacobian_contacts: scratch must be 256 B aligned");
  const long long PA = (long long)P * A;
  uint8_t* s = (uint8_t*)scratch;
  double* Jc = reinterpret_cast<double*>(s);
  double* F = reinterpret_cast<double*>(s + align256_((size_t)PA * PA * 8));
  double* sums = reinterpret_cast<double*>(s + align256_((size_t)PA * PA * 8) + align256_((size_t)P * P * 8));
  // centre over i, a, j, b in turn: [outer, n, inner] = [1, P, A*P*A], [P, A, P*A], [P*A, P, A], [P*A*P, A, 1]
  jacobian_center_kernel<float><<<grid_blocks(PA * A), 256, 0, st>>>(J, Jc, 1, P, PA * A);
  jacobian_center_kernel<double><<<grid_blocks(PA * P), 256, 0, st>>>(Jc, Jc, P, A, PA);
  jacobian_center_kernel<double><<<grid_blocks(PA * A), 256, 0, st>>>(Jc, Jc, PA, P, A);
  jacobian_center_kernel<double><<<grid_blocks(PA * P), 256, 0, st>>>(Jc, Jc, PA * P, A, 1);
  jacobian_frobenius_kernel<<<grid_blocks((long long)P * P), 256, 0, st>>>(Jc, P, A, F);
  count_launch(5);
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return launch_apc_contacts(F, P, sums, contacts_out, st);
}

}  // extern "C"
