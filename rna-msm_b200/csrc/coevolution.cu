// Statistics of an alignment itself, on every row of it: sequence weights, Neff and mean-field DCA contacts
// (Morcos et al., PNAS 2011).  tests/dca_ref.py restates every step in float64 numpy.
//
//   tokens int64 [N, C], column 0 BOS, residues 1 .. L = C - 1
//   states   s[n, l] = tokens[n, l + 1] - 4 for A G C U (vocabulary 4 .. 7), else 4 (the gap state); q = 5
//   weights  row k is a neighbour of row n iff (double) m(n, k) >= theta * (double) L, m = number of equal states
//            (gap == gap counts); w[n] = 1.0 / count[n]; Neff = sum_n w[n]
//   freqs    f_i(a) = (1 - lam) / Neff * sum_n w_n [s_ni = a] + lam / q
//            f_ij(a, b) = (1 - lam) / Neff * sum_n w_n [s_ni = a][s_nj = b] + lam / q^2 (i != j), f_ii(a, b) = f_i(a) d_ab
//   Cov      [(i, a), (j, b)] = f_ij(a, b) - f_i(a) f_j(b), a, b < 4 (gap state dropped): side M = 4L
//   e        -Cov^-1 by a blocked Cholesky factorisation Cov = L L^T, L^-1, then Cov^-1 = L^-T L^-1
//   scores   F[i, j] = Frobenius norm of the 4 x 4 block e_ij padded to 5 x 5 with zeros and put in the zero-sum
//            gauge; F[i, i] = 0; then the APC and symmetrisation of rnamsm_jacobian_contacts
//
// Every reduction is a loop in a fixed order (no atomics), so repeated calls give the same bits.
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

constexpr int kQ = 5;          // states: A G C U and the gap state
constexpr int kWordStates = 8; // 4-bit states per packed uint32
constexpr int kNB = 64;        // block size of the Cholesky factorisation and inverse
constexpr int kCountKT = 32;   // rows k per shared tile of the neighbour count
constexpr int kCountWC = 8;    // packed words per chunk of the neighbour count
constexpr int kPotrfSmem = 2 * kNB * (kNB + 1) * 8;

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
static __host__ __device__ int packed_words(int L) { return (L + kWordStates - 1) / kWordStates; }
static int padded_side(int L) { return ((4 * L + kNB - 1) / kNB) * kNB; }

// The neighbour count splits the k range into this many slices when the n rows alone would not fill the GPU.
static int count_splits(int N) {
  const int bx = ceil_div(N, 256);
  const int want = std::max(1, ceil_div(2 * 148, bx));
  return std::min(want, ceil_div(N, kCountKT));
}
static int count_chunk(int N, int S) { return ceil_div(ceil_div(N, S), kCountKT) * kCountKT; }

// Smallest integer m with (double) m >= theta * (double) L; rows with at most L - that many mismatches are neighbours.
static int max_mismatches(int L, double theta) {
  const double t = theta * (double)L;
  return L - (int)ceil(t);
}

struct WeightsLayout {
  size_t packed, partial, total;
};
static WeightsLayout weights_layout(int N, int L) {
  WeightsLayout w;
  w.packed = 0;
  w.partial = align256((size_t)N * packed_words(L) * 4);
  w.total = w.partial + align256((size_t)count_splits(N) * N * 4);
  return w;
}

// DCA workspace: status int32 | weights workspace | states uint8 [N, L] | fi double [L, 4] | buffer A double [Mp, Mp]
// (Cov, then L, then e) | buffer B double [Mp, Mp] (L^-1) | F double [L, L] | sums double [2L + 1]
struct DcaLayout {
  size_t weights, states, fi, a, b, F, sums, total;
};
static DcaLayout dca_layout(int N, int L) {
  const size_t Mp = padded_side(L);
  DcaLayout d;
  d.weights = 256;
  d.states = d.weights + weights_layout(N, L).total;
  d.fi = d.states + align256((size_t)N * L);
  d.a = d.fi + align256((size_t)L * 4 * 8);
  d.b = d.a + align256(Mp * Mp * 8);
  d.F = d.b + align256(Mp * Mp * 8);
  d.sums = d.F + align256((size_t)L * L * 8);
  d.total = d.sums + align256((2 * (size_t)L + 1) * 8);
  return d;
}

static int grid_for(long long total) { return (int)std::min<long long>((total + 255) / 256, 148LL * 16); }

static __device__ __forceinline__ int token_state(int64_t t) { return (t >= 4 && t <= 7) ? (int)(t - 4) : 4; }

// ------------------------------------------------------------------------------------------------ states
// One thread per (row, packed word): 8 states as nibbles (columns past L hold 0 in every row, so they never differ);
// with `states` the uint8 grid [N, L] as well.
__global__ void __launch_bounds__(256)
dca_states_kernel(const int64_t* __restrict__ tokens, int N, int C, uint32_t* __restrict__ packed,
                  uint8_t* __restrict__ states) {
  const int L = C - 1, W = packed_words(L);
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)N * W;
       e += (long long)gridDim.x * blockDim.x) {
    const long long n = e / W;
    const int w = (int)(e - n * W);
    uint32_t word = 0;
    for (int q = 0; q < kWordStates; ++q) {
      const int l = w * kWordStates + q;
      if (l < L) {
        const int s = token_state(tokens[n * C + 1 + l]);
        word |= (uint32_t)s << (4 * q);
        if (states) states[n * L + l] = (uint8_t)s;
      }
    }
    packed[e] = word;
  }
}

// ------------------------------------------------------------------------------------------------ neighbour counts
// partial[y, n] = number of rows k in slice y (rows [y * chunk, (y + 1) * chunk)) with at most maxmis mismatching
// states against row n.  XOR of two packed words leaves a nonzero nibble (<= 7) where the states differ; adding 7 to
// every nibble carries into its top bit exactly then, and popc counts those bits.  Each thread owns one row n; a
// tile of kCountKT rows k is staged in shared memory kCountWC words at a time and read as a broadcast.
__global__ void __launch_bounds__(256)
dca_neighbour_count_kernel(const uint32_t* __restrict__ packed, int N, int W, int maxmis, int chunk,
                           int* __restrict__ partial) {
  __shared__ __align__(16) uint32_t sk[kCountKT][kCountWC];
  const int tid = threadIdx.x;
  const int n = blockIdx.x * 256 + tid;
  const int kb = blockIdx.y * chunk, ke = min(N, kb + chunk);
  int count = 0;
  for (int k0 = kb; k0 < ke; k0 += kCountKT) {
    int mis[kCountKT];
#pragma unroll
    for (int kk = 0; kk < kCountKT; ++kk) mis[kk] = 0;
    for (int w0 = 0; w0 < W; w0 += kCountWC) {
      __syncthreads();
      {
        const int kk = tid / kCountWC, w = tid % kCountWC;
        sk[kk][w] = (k0 + kk < ke && w0 + w < W) ? packed[(long long)(k0 + kk) * W + w0 + w] : 0u;
      }
      __syncthreads();
      uint32_t my[kCountWC];
#pragma unroll
      for (int w = 0; w < kCountWC; ++w) my[w] = (n < N && w0 + w < W) ? packed[(long long)n * W + w0 + w] : 0u;
#pragma unroll
      for (int kk = 0; kk < kCountKT; ++kk) {
        int m = 0;
#pragma unroll
        for (int w = 0; w < kCountWC; ++w) m += __popc(((my[w] ^ sk[kk][w]) + 0x77777777u) & 0x88888888u);
        mis[kk] += m;
      }
    }
#pragma unroll
    for (int kk = 0; kk < kCountKT; ++kk) count += (k0 + kk < ke && mis[kk] <= maxmis) ? 1 : 0;
  }
  if (n < N) partial[(long long)blockIdx.y * N + n] = count;
}

// w[n] = 1.0 / (sum of the slices' counts); neff[0] = sum_n w[n]: each thread adds its rows t, t + 1024, ... in
// ascending order, then a fixed tree over the threads.  One block of 1024 threads.
__global__ void __launch_bounds__(1024)
dca_weights_kernel(const int* __restrict__ partial, int S, int N, double* __restrict__ w, double* __restrict__ neff) {
  __shared__ double red[1024];
  double s = 0.0;
  for (int n = threadIdx.x; n < N; n += 1024) {
    int c = 0;
    for (int y = 0; y < S; ++y) c += partial[(long long)y * N + n];
    const double v = 1.0 / (double)c;
    w[n] = v;
    s += v;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int h = 512; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) neff[0] = red[0];
}

// ------------------------------------------------------------------------------------------------ frequencies, Cov
// One thread per column i: fi[i, a] and the diagonal block Cov[(i, a), (i, b)] = f_i(a) d_ab - f_i(a) f_i(b).
// Rows M .. Mp - 1 of the padded matrix get the identity (lower triangle), so it factors block by block.
__global__ void __launch_bounds__(256)
dca_sites_kernel(const uint8_t* __restrict__ states, const double* __restrict__ w, const double* __restrict__ neff, int N,
                 int L, double lam, double* __restrict__ fi, double* __restrict__ A, int Mp) {
  const double c1 = (1.0 - lam) / neff[0];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) {
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int n = 0; n < N; ++n) {
      const int s = states[(long long)n * L + i];
      const double v = w[n];
#pragma unroll
      for (int a = 0; a < 4; ++a) acc[a] += s == a ? v : 0.0;
    }
    double f[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      f[a] = c1 * acc[a] + lam / kQ;
      fi[i * 4 + a] = f[a];
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) A[(long long)(4 * i + a) * Mp + 4 * i + b] = (a == b ? f[a] : 0.0) - f[a] * f[b];
  }
  const int M = 4 * L;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)(Mp - M) * Mp;
       e += (long long)gridDim.x * blockDim.x) {
    const long long r = M + e / Mp, c = e % Mp;
    A[r * Mp + c] = r == c ? 1.0 : 0.0;
  }
}

// Pair counts, output-stationary: block (j-tile, i) and its thread j > i own the 16 bins (a, b < 4) of the pair,
// kept in shared memory as bins[ab][thread] and summed over n ascending.  The lower-triangle entries
// Cov[(j, b), (i, a)] = f_ij(a, b) - f_i(a) f_j(b) are written straight from them.
__global__ void __launch_bounds__(256)
dca_pairs_kernel(const uint8_t* __restrict__ states, const double* __restrict__ w, const double* __restrict__ neff,
                 const double* __restrict__ fi, int N, int L, double lam, double* __restrict__ A, int Mp) {
  __shared__ double bins[16][256];
  const int tid = threadIdx.x;
  const int j = blockIdx.x * 256 + tid;
  const double c1 = (1.0 - lam) / neff[0];
  for (int i = blockIdx.y; i < L; i += gridDim.y) {
    if (i >= blockIdx.x * 256 + 255) continue;  // block-uniform: no j of this block is past i
#pragma unroll
    for (int ab = 0; ab < 16; ++ab) bins[ab][tid] = 0.0;
    const bool own = j > i && j < L;
    if (own) {
      for (int n = 0; n < N; ++n) {
        const int a = states[(long long)n * L + i], b = states[(long long)n * L + j];
        if (a < 4 && b < 4) bins[a * 4 + b][tid] += w[n];
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
          A[(long long)(4 * j + b) * Mp + 4 * i + a] = (c1 * bins[a * 4 + b][tid] + lam / (kQ * kQ)) - fi[i * 4 + a] * fi[j * 4 + b];
    }
  }
}

// ------------------------------------------------------------------------------------------------ Cholesky, inverse
// acc[u][v] += sum_p opA(r, p) opB(p, c) over one 64 x 64 x 64 tile product, r = ty + 16u, c = tx + 16v (256
// threads as 16 x 16).  opA(r, p) = A[r * ld + p] (TA: A[p * ld + r]); opB(p, c) = B[p * ld + c] (TB: B[c * ld + p]).
// The k axis is staged 16 wide through shared memory, in ascending order.
template <bool TA, bool TB>
__device__ __forceinline__ void tile_mma(const double* __restrict__ A, const double* __restrict__ B, long long ld,
                                         double (&sA)[kNB][17], double (&sB)[16][kNB + 1], double (&acc)[4][4]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int k0 = 0; k0 < kNB; k0 += 16) {
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + 256 * q;
      if (TA) {
        const int r = e & 63, p = e >> 6;
        sA[r][p] = A[(long long)(k0 + p) * ld + r];
      } else {
        const int r = e >> 4, p = e & 15;
        sA[r][p] = A[(long long)r * ld + k0 + p];
      }
      if (TB) {
        const int c = e >> 4, p = e & 15;
        sB[p][c] = B[(long long)c * ld + k0 + p];
      } else {
        const int c = e & 63, p = e >> 6;
        sB[p][c] = B[(long long)(k0 + p) * ld + c];
      }
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 16; ++p) {
      double a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] = sA[ty + 16 * u][p];
#pragma unroll
      for (int v = 0; v < 4; ++v) b[v] = sB[p][tx + 16 * v];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fma(a[u], b[v], acc[u][v]);
    }
  }
}

static __device__ __forceinline__ double* blk(double* X, int Mp, int bi, int bj) {
  return X + (long long)bi * kNB * Mp + (long long)bj * kNB;
}

// Diagonal block kk: Cholesky of its lower triangle in shared memory into A (upper part zeroed), and the inverse of that
// triangle into the diagonal block of B (upper part zeroed: it is the diagonal block of L^-1).  A pivot that is not
// positive sets *status = 1 + its index (the first one only) and continues as NaN.
__global__ void __launch_bounds__(256)
dca_potrf_diag_kernel(double* __restrict__ A, double* __restrict__ B, int Mp, int kk, int* __restrict__ status) {
  extern __shared__ double smem_diag[];  // kPotrfSmem bytes: a and x, [kNB][kNB + 1] each
  double (*a)[kNB + 1] = reinterpret_cast<double (*)[kNB + 1]>(smem_diag);
  double (*x)[kNB + 1] = reinterpret_cast<double (*)[kNB + 1]>(smem_diag + kNB * (kNB + 1));
  const int tid = threadIdx.x;
  double* Ad = blk(A, Mp, kk, kk);
  double* Bd = blk(B, Mp, kk, kk);
  for (int e = tid; e < kNB * kNB; e += 256) a[e / kNB][e % kNB] = Ad[(long long)(e / kNB) * Mp + e % kNB];
  __syncthreads();
  for (int j = 0; j < kNB; ++j) {
    if (tid == 0) {
      const double d = a[j][j];
      if (!(d > 0.0)) {
        if (*status == 0) *status = 1 + kk * kNB + j;
        a[j][j] = nan("");
      } else {
        a[j][j] = sqrt(d);
      }
    }
    __syncthreads();
    for (int r = j + 1 + tid; r < kNB; r += 256) a[r][j] /= a[j][j];
    __syncthreads();
    const int m = kNB - 1 - j;  // trailing rows / columns j + 1 .. 63
    for (int e = tid; e < m * m; e += 256) {
      const int r = j + 1 + e / m, c = j + 1 + e % m;
      if (c <= r) a[r][c] -= a[r][j] * a[c][j];
    }
    __syncthreads();
  }
  // inverse of the lower triangle, one thread per column c: x[r][c] = (d_rc - sum_{p<r} a[r][p] x[p][c]) / a[r][r]
  if (tid < kNB) {
    const int c = tid;
    for (int r = 0; r < kNB; ++r) {
      double v = 0.0;
      if (r >= c) {
        double s = r == c ? 1.0 : 0.0;
        for (int p = c; p < r; ++p) s -= a[r][p] * x[p][c];
        v = s / a[r][r];
      }
      x[r][c] = v;
    }
  }
  __syncthreads();
  for (int e = tid; e < kNB * kNB; e += 256) {
    const int r = e / kNB, c = e % kNB;
    Ad[(long long)r * Mp + c] = c <= r ? a[r][c] : 0.0;
    Bd[(long long)r * Mp + c] = x[r][c];
  }
}

// Panel: L[i][kk] = A[i][kk] (L[kk][kk])^-T for the block rows i > kk, one block row per CTA.
__global__ void __launch_bounds__(256)
dca_potrf_panel_kernel(double* __restrict__ A, const double* __restrict__ B, int Mp, int kk) {
  __shared__ double sA[kNB][17];
  __shared__ double sB[16][kNB + 1];
  const int i = kk + 1 + blockIdx.x;
  double acc[4][4] = {};
  double* Ai = blk(A, Mp, i, kk);
  tile_mma<false, true>(Ai, blk(const_cast<double*>(B), Mp, kk, kk), Mp, sA, sB, acc);
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) Ai[(long long)(ty + 16 * u) * Mp + tx + 16 * v] = acc[u][v];
}

// lower-triangle block pair number t -> (i, j), j <= i, of a triangle whose first block is `base`
static __device__ __forceinline__ void tri_index(int t, int base, int& i, int& j) {
  int r = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((r + 1) * (r + 2) / 2 <= t) ++r;
  while (r * (r + 1) / 2 > t) --r;
  i = base + r;
  j = base + t - r * (r + 1) / 2;
}

// Trailing update: A[i][j] -= L[i][kk] L[j][kk]^T for the lower blocks kk < j <= i.
__global__ void __launch_bounds__(256)
dca_potrf_update_kernel(double* __restrict__ A, int Mp, int kk) {
  __shared__ double sA[kNB][17];
  __shared__ double sB[16][kNB + 1];
  int i, j;
  tri_index(blockIdx.x, kk + 1, i, j);
  double acc[4][4] = {};
  tile_mma<false, true>(blk(A, Mp, i, kk), blk(A, Mp, j, kk), Mp, sA, sB, acc);
  double* Aij = blk(A, Mp, i, j);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) Aij[(long long)(ty + 16 * u) * Mp + tx + 16 * v] -= acc[u][v];
}

// Off-diagonal blocks of L^-1 at block distance d: for i = j + d,
//   B[i][j] = -B[i][i] sum_{k=j}^{i-1} L[i][k] B[k][j]
// The blocks a launch reads are at distances < d, so one launch per d.  The partial sum goes through B[i][j] itself.
__global__ void __launch_bounds__(256)
dca_trtri_kernel(const double* __restrict__ A, double* __restrict__ B, int Mp, int d) {
  __shared__ double sA[kNB][17];
  __shared__ double sB[16][kNB + 1];
  const int j = blockIdx.x, i = j + d;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4] = {};
  for (int k = j; k < i; ++k)
    tile_mma<false, false>(blk(const_cast<double*>(A), Mp, i, k), blk(B, Mp, k, j), Mp, sA, sB, acc);
  double* Bij = blk(B, Mp, i, j);
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) Bij[(long long)(ty + 16 * u) * Mp + tx + 16 * v] = acc[u][v];
  __syncthreads();
  double out[4][4] = {};
  tile_mma<false, false>(blk(B, Mp, i, i), Bij, Mp, sA, sB, out);
  __syncthreads();
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) Bij[(long long)(ty + 16 * u) * Mp + tx + 16 * v] = -out[u][v];
}

// e = -Cov^-1 = -(L^-1)^T L^-1 into A: block (i, j), j <= i, is -sum_{k >= i} B[k][i]^T B[k][j]; it and its transpose
// are written.  The diagonal blocks come out symmetric bit for bit (the same products summed in the same order).
__global__ void __launch_bounds__(256)
dca_lauum_kernel(const double* __restrict__ B, double* __restrict__ A, int Mp) {
  __shared__ double sA[kNB][17];
  __shared__ double sB[16][kNB + 1];
  const int T = Mp / kNB;
  int i, j;
  tri_index(blockIdx.x, 0, i, j);
  double acc[4][4] = {};
  for (int k = i; k < T; ++k)
    tile_mma<true, false>(blk(const_cast<double*>(B), Mp, k, i), blk(const_cast<double*>(B), Mp, k, j), Mp, sA, sB, acc);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double* Aij = blk(A, Mp, i, j);
  double* Aji = blk(A, Mp, j, i);
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int r = ty + 16 * u, c = tx + 16 * v;
      Aij[(long long)r * Mp + c] = -acc[u][v];
      Aji[(long long)c * Mp + r] = -acc[u][v];
    }
}

// ------------------------------------------------------------------------------------------------ scores
// F[i, j] = || gauge(pad(e_ij)) ||_F for i != j, 0 on the diagonal; e_ij padded with a zero row and column (the gap
// state), then row means and column means subtracted and the overall mean added back.
__global__ void __launch_bounds__(256)
dca_scores_kernel(const double* __restrict__ E, int Mp, int L, double* __restrict__ F) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)L * L;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / L), j = (int)(e - (long long)i * L);
    if (i == j) {
      F[e] = 0.0;
      continue;
    }
    double x[kQ][kQ];
#pragma unroll
    for (int a = 0; a < kQ; ++a)
#pragma unroll
      for (int b = 0; b < kQ; ++b) x[a][b] = (a < 4 && b < 4) ? E[(long long)(4 * i + a) * Mp + 4 * j + b] : 0.0;
    double rm[kQ], cm[kQ], all = 0.0;
#pragma unroll
    for (int a = 0; a < kQ; ++a) {
      double s = 0.0;
#pragma unroll
      for (int b = 0; b < kQ; ++b) s += x[a][b];
      rm[a] = s / kQ;
    }
#pragma unroll
    for (int b = 0; b < kQ; ++b) {
      double s = 0.0;
#pragma unroll
      for (int a = 0; a < kQ; ++a) s += x[a][b];
      cm[b] = s / kQ;
    }
#pragma unroll
    for (int a = 0; a < kQ; ++a) all += rm[a];
    all /= kQ;
    double s = 0.0;
#pragma unroll
    for (int a = 0; a < kQ; ++a)
#pragma unroll
      for (int b = 0; b < kQ; ++b) {
        const double v = x[a][b] - rm[a] - cm[b] + all;
        s += v * v;
      }
    F[e] = sqrt(s);
  }
}

static int check_tokens(const void* tokens, int N, int C, const char* who) {
  RNAMSM_REQUIRE(tokens, "%s: tokens required", who);
  RNAMSM_REQUIRE(N >= 1 && C >= 2, "%s: need N >= 1 rows and L = C - 1 >= 1 residues (N=%d C=%d)", who, N, C);
  return 0;
}

// states, neighbour counts, weights and Neff (4 launches); `ws` holds weights_layout(N, L)
static int seq_weights(const int64_t* tokens, int N, int C, double theta, double* w, double* neff, uint8_t* ws,
                uint8_t* states, int* launches, cudaStream_t st) {
  const int L = C - 1, W = packed_words(L);
  const WeightsLayout lay = weights_layout(N, L);
  uint32_t* packed = reinterpret_cast<uint32_t*>(ws + lay.packed);
  int* partial = reinterpret_cast<int*>(ws + lay.partial);
  const int S = count_splits(N), chunk = count_chunk(N, S);
  dca_states_kernel<<<grid_for((long long)N * W), 256, 0, st>>>(tokens, N, C, packed, states);
  dca_neighbour_count_kernel<<<dim3(ceil_div(N, 256), S), 256, 0, st>>>(packed, N, W, max_mismatches(L, theta), chunk,
                                                                       partial);
  dca_weights_kernel<<<1, 1024, 0, st>>>(partial, S, N, w, neff);
  *launches += 3;
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

size_t rnamsm_seq_weights_workspace_bytes(int N, int L) {
  if (N < 1 || L < 1) {
    set_error("seq_weights: need N >= 1 rows and L >= 1 residues (N=%d L=%d)", N, L);
    return 0;
  }
  return weights_layout(N, L).total;
}

int rnamsm_msa_seq_weights(const int64_t* tokens, int N, int C, double theta, double* weights_out, double* neff_out,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_tokens(tokens, N, C, "seq_weights")) return rc;
  RNAMSM_REQUIRE(theta > 0.0 && theta <= 1.0, "seq_weights: theta %g outside (0, 1]", theta);
  RNAMSM_REQUIRE(weights_out && neff_out && workspace, "seq_weights: weights_out, neff_out and workspace required");
  const size_t need = weights_layout(N, C - 1).total;
  RNAMSM_REQUIRE(workspace_bytes >= need, "seq_weights: workspace %zu < required %zu", workspace_bytes, need);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "seq_weights: workspace must be 256 B aligned");
  int launches = 0;
  const int rc = seq_weights(tokens, N, C, theta, weights_out, neff_out, (uint8_t*)workspace, nullptr, &launches,
                             (cudaStream_t)stream);
  count_launch(launches);
  return rc;
}

size_t rnamsm_dca_workspace_bytes(int N, int L) {
  if (N < 1 || L < 1) {
    set_error("dca: need N >= 1 rows and L >= 1 residues (N=%d L=%d)", N, L);
    return 0;
  }
  return dca_layout(N, L).total;
}

int rnamsm_msa_dca(const int64_t* tokens, int N, int C, double theta, double pseudocount, double* weights_out,
                   double* neff_out, float* contacts_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_tokens(tokens, N, C, "dca")) return rc;
  RNAMSM_REQUIRE(theta > 0.0 && theta <= 1.0, "dca: theta %g outside (0, 1]", theta);
  RNAMSM_REQUIRE(pseudocount > 0.0 && pseudocount < 1.0, "dca: pseudocount %g outside (0, 1)", pseudocount);
  RNAMSM_REQUIRE(weights_out && neff_out && contacts_out && workspace,
                 "dca: weights_out, neff_out, contacts_out and workspace required");
  const int L = C - 1;
  const DcaLayout lay = dca_layout(N, L);
  RNAMSM_REQUIRE(workspace_bytes >= lay.total, "dca: workspace %zu < required %zu", workspace_bytes, lay.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "dca: workspace must be 256 B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  int* status = reinterpret_cast<int*>(ws);
  uint8_t* states = ws + lay.states;
  double* fi = reinterpret_cast<double*>(ws + lay.fi);
  double* A = reinterpret_cast<double*>(ws + lay.a);
  double* B = reinterpret_cast<double*>(ws + lay.b);
  double* F = reinterpret_cast<double*>(ws + lay.F);
  double* sums = reinterpret_cast<double*>(ws + lay.sums);
  const int Mp = padded_side(L), T = Mp / kNB;
  int launches = 0;
  RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(dca_potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPotrfSmem));
  RNAMSM_CHECK_CUDA(cudaMemsetAsync(status, 0, sizeof(int), st));
  if (int rc = seq_weights(tokens, N, C, theta, weights_out, neff_out, ws + lay.weights, states, &launches, st)) return rc;
  dca_sites_kernel<<<grid_for(std::max<long long>(L, (long long)(Mp - 4 * L) * Mp)), 256, 0, st>>>(
      states, weights_out, neff_out, N, L, pseudocount, fi, A, Mp);
  dca_pairs_kernel<<<dim3(ceil_div(L, 256), std::min(L, 65535)), 256, 0, st>>>(states, weights_out, neff_out, fi, N, L,
                                                                              pseudocount, A, Mp);
  launches += 2;
  for (int kk = 0; kk < T; ++kk) {
    dca_potrf_diag_kernel<<<1, 256, kPotrfSmem, st>>>(A, B, Mp, kk, status);
    ++launches;
    const int rest = T - 1 - kk;
    if (rest > 0) {
      dca_potrf_panel_kernel<<<rest, 256, 0, st>>>(A, B, Mp, kk);
      dca_potrf_update_kernel<<<rest * (rest + 1) / 2, 256, 0, st>>>(A, Mp, kk);
      launches += 2;
    }
  }
  for (int d = 1; d < T; ++d) {
    dca_trtri_kernel<<<T - d, 256, 0, st>>>(A, B, Mp, d);
    ++launches;
  }
  dca_lauum_kernel<<<T * (T + 1) / 2, 256, 0, st>>>(B, A, Mp);
  dca_scores_kernel<<<grid_for((long long)L * L), 256, 0, st>>>(A, Mp, L, F);
  launches += 2;
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  count_launch(launches);
  return launch_apc_contacts(F, L, sums, contacts_out, st);
}

}  // extern "C"
