// Nested secondary structure from a pair map: maximum expected accuracy folding ("mea") or maximum-weight nested
// matching ("score").  tests/fold_ref.py restates it in float32 numpy; the device result is bit-identical to it.
//
//   allowed  (i, k), i < k: k - i > min_loop, S[i, k] > threshold, and with canonical {s_i, s_k} in {AU, GC, GU}
//   weights  mea: w[i, k] = fp32(2 gamma) * S[i, k], u[i] = fp32(1 - sum_{j != i} S[min, max]) (float64, ascending j)
//            score: w[i, k] = S[i, k], u[i] = 0
//   P[i][k]  = w[i, k] + M[i+1][k-1] if (i, k) is allowed, else -inf      (M[a][a-1] = 0: the empty interval)
//   M[i][j]  = max(M[i+1][j] + u[i], max_{i < k <= j} P[i][k] + M[k+1][j])
//
// Every candidate is one fp32 add of two stored values and max is exact, so the tables do not depend on the order in
// which the candidates are visited: not on the tiling, the split of the bulk range, or the batch.
//
// Tables, per map: M [Lp, ld] and P [Lp, ld] (Lp = L rounded up to the tile T, ld = Lp + 4).  P[i][k] is stored at
// column k + 1, so that the candidate P[i][k] + M[k+1][j] reads column c = k + 1 of P and row c of M: the bulk of the
// recurrence is the tropical product max_c P'[i][c] + M[c][j].  The prep kernel stores w (or -inf) where P goes; the
// fill overwrites each allowed entry with P when it reaches it.
#include <limits.h>
#include <math.h>

#include <algorithm>
#include <vector>

#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

constexpr int kFoldThreads = 256;
constexpr int kFoldKT = 16;           // inner slice of the bulk product staged per step
constexpr int kFoldTargetCTAs = 296;  // 2 per SM of a 148-SM B200; the split uses this constant, not the device
constexpr int kFoldMaxL = 1 << 20;
constexpr int kFoldMaxMaps = 65535;   // gridDim.y of the prep kernel

struct FoldMap {
  const float* S;      // [L, L], upper triangle read
  const uint8_t* seq;  // [L] codes 0..3 = A G C U, anything else never pairs; null without canonical
  int* pairs;          // [L] out
  float* M;            // [Lp, ld]
  float* P;            // [Lp, ld], P[i][k] at column k + 1
  float* u;            // [Lp]
  int* stack;          // [2 L + 2] intervals of the traceback
  int L, Lp, ld, nt;   // nt = Lp / T tiles per side
  int ntpre;           // sum of nt over the maps before this one (descriptors sorted by nt, descending)
  int out;             // index into scores_out
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Tile side: 32 while every map is at most 1024 long (half the serial steps of each in-tile row), else 64.
static int fold_tile(int Lmax) { return Lmax <= 1024 ? 32 : 64; }

// CTAs sharing one tile's bulk range on diagonal delta, from the shape only: enough to give kFoldTargetCTAs CTAs in
// all, at least one T-wide slice of the range each.
static int fold_splits(int delta, long long tiles) {
  if (delta < 2) return 1;
  return (int)std::min<long long>(delta - 1, (kFoldTargetCTAs + tiles - 1) / tiles);
}

struct FoldPlan {
  int T = 0, ntmax = 0;
  std::vector<int> order;  // map indices sorted by L, descending (stable)
  std::vector<int> nt;     // per map, in call order
  size_t desc = 0, counters = 0, partial = 0, total = 0;
  std::vector<size_t> u, stack, M, P;  // per map, in call order
  std::vector<long long> tiles;        // per diagonal
};

static size_t fold_table_bytes(int Lp) { return align256((size_t)Lp * (Lp + 4) * 4); }

// Workspace: flag int32 (256 B) | descriptors | tile counters (one per tile of diagonal 0) | split-K partials |
// per map: u, stack, M, P.
static int fold_plan(int n, const int* L, FoldPlan& p) {
  RNAMSM_REQUIRE(n >= 1 && n <= kFoldMaxMaps, "fold: need 1 <= n <= %d maps, got %d", kFoldMaxMaps, n);
  RNAMSM_REQUIRE(L, "fold: L required");
  int Lmax = 0;
  for (int m = 0; m < n; ++m) {
    RNAMSM_REQUIRE(L[m] >= 1 && L[m] <= kFoldMaxL, "fold: map %d has L = %d, outside [1, %d]", m, L[m], kFoldMaxL);
    Lmax = std::max(Lmax, L[m]);
  }
  p.T = fold_tile(Lmax);
  p.ntmax = ceil_div(Lmax, p.T);
  p.nt.resize(n);
  long long ntsum = 0;
  for (int m = 0; m < n; ++m) {
    p.nt[m] = ceil_div(L[m], p.T);
    ntsum += p.nt[m];
  }
  p.order.resize(n);
  for (int m = 0; m < n; ++m) p.order[m] = m;
  std::stable_sort(p.order.begin(), p.order.end(), [&](int a, int b) { return p.nt[a] > p.nt[b]; });
  p.tiles.assign(p.ntmax, 0);
  size_t partial = 0;
  for (int d = 0; d < p.ntmax; ++d) {
    for (int m = 0; m < n; ++m) p.tiles[d] += std::max(0, p.nt[m] - d);
    const int S = fold_splits(d, p.tiles[d]);
    if (S > 1) partial = std::max(partial, (size_t)p.tiles[d] * S * p.T * p.T * 4);
  }
  p.desc = 256;
  p.counters = p.desc + align256((size_t)n * sizeof(FoldMap));
  p.partial = p.counters + align256((size_t)ntsum * 4);
  size_t off = p.partial + align256(partial);
  p.u.resize(n), p.stack.resize(n), p.M.resize(n), p.P.resize(n);
  for (int m = 0; m < n; ++m) {
    const int Lp = p.nt[m] * p.T;
    p.u[m] = off;
    off += align256((size_t)Lp * 4);
    p.stack[m] = off;
    off += align256((2 * (size_t)L[m] + 2) * 4);
    p.M[m] = off;
    off += fold_table_bytes(Lp);
    p.P[m] = off;
    off += fold_table_bytes(Lp);
  }
  p.total = off;
  return 0;
}

static __device__ __forceinline__ bool canonical_pair(int a, int b) {
  // A G C U = 0 1 2 3: AU, UA, GC, CG, GU, UG
  constexpr unsigned kOk = (1u << (0 * 4 + 3)) | (1u << (3 * 4 + 0)) | (1u << (1 * 4 + 2)) | (1u << (2 * 4 + 1)) |
                           (1u << (1 * 4 + 3)) | (1u << (3 * 4 + 1));
  return a < 4 && b < 4 && ((kOk >> (a * 4 + b)) & 1u);
}

// ------------------------------------------------------------------------------------------------ prep
// blockIdx.y = map.  Every entry of the map's P table: w of an allowed pair at column k + 1, -inf elsewhere (padding
// included).  u for every row (0 past L).  flag bits: 1 for a non-finite entry of the upper triangle, 2 for a weight
// or a u that overflows.  Block (0, 0) also clears the tile counters of the split-K combine.
__global__ void __launch_bounds__(kFoldThreads)
fold_prep_kernel(const FoldMap* __restrict__ maps, int mea, float g, float thr, int min_loop, int canonical,
                 int* __restrict__ flag, int* __restrict__ counters, int ncounters) {
  const FoldMap mp = maps[blockIdx.y];
  const int L = mp.L, ld = mp.ld, tid = threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + tid;
  if (blockIdx.y == 0)
    for (long long e = t0; e < ncounters; e += stride) counters[e] = 0;
  for (int i = blockIdx.x; i < mp.Lp; i += gridDim.x) {
    float* __restrict__ row = mp.P + (long long)i * ld;
    for (int c = tid; c < ld; c += blockDim.x) {
      const int k = c - 1;
      float v = -INFINITY;
      if (i < L && k > i && k < L) {
        const float s = mp.S[(long long)i * L + k];
        if (!isfinite(s)) atomicOr(flag, 1);
        const bool ok = k - i > min_loop && s > thr && (!canonical || canonical_pair(mp.seq[i], mp.seq[k]));
        if (ok) {
          v = mea ? g * s : s;
          if (isfinite(s) && !isfinite(v)) atomicOr(flag, 2);
        }
      }
      row[c] = v;
    }
  }
  for (long long i = t0; i < mp.Lp; i += stride) {
    float u = 0.f;
    if (mea && i < L) {
      double acc = 0.0;
      for (int j = 0; j < L; ++j)
        if (j != i) acc += (double)(j < i ? mp.S[(long long)j * L + i] : mp.S[i * L + j]);
      u = (float)(1.0 - acc);
      if (isfinite(acc) && !isfinite(u)) atomicOr(flag, 2);
    }
    mp.u[i] = u;
  }
}

// ------------------------------------------------------------------------------------------------ fill
template <int T>
constexpr int fold_fill_smem() {
  return (4 * T * (T + 1) + (T + 1) + 3 * T + kFoldKT * (T + 4) + kFoldKT * T) * 4;
}

template <int N>
static __device__ __forceinline__ void lds_vec(float (&r)[N], const float* p) {
  if constexpr (N == 4) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    r[0] = v.x, r[1] = v.y, r[2] = v.z, r[3] = v.w;
  } else {
    const float2 v = *reinterpret_cast<const float2*>(p);
    r[0] = v.x, r[1] = v.y;
  }
}

// One launch per tile diagonal delta.  blockIdx.x = slot * S + s: slot numbers the tiles (I, J = I + delta) of every
// map that has this diagonal (maps in descriptor order, I ascending), s the slice of the bulk range.
//   (a) bulk: B[i][j] = max_{c in slice} P'[i][c] + M[c][j] over c in [(I+1) T, J T), whose operands lie in tiles of
//       earlier diagonals; register-tiled like an SGEMM (TM x TM cells a thread, FADD + FMNMX), operands staged
//       through shared memory.  With S > 1 each slice writes its partial maximum and the last CTA of the tile to
//       arrive combines them and goes on alone.
//   (b) in-tile: rows bottom-up; for each row first P of the row's T columns (it needs row i + 1 of M only), then M of
//       the row's T cells, G = 256 / T threads per cell splitting the remaining candidates, combined with shuffles.
template <int T>
__global__ void __launch_bounds__(kFoldThreads)
fold_fill_kernel(const FoldMap* __restrict__ maps, int count, int delta, int S, float* __restrict__ partial,
                 int* __restrict__ counters) {
  constexpr int G = kFoldThreads / T;
  constexpr int TM = T / 16;
  constexpr int SP = T + 1;
  constexpr int AP = T + 4;
  constexpr int KT = kFoldKT;
  extern __shared__ __align__(16) float smf[];
  float* Mc = smf;              // [T][SP] this tile of M
  float* Md = Mc + T * SP;      // [T][SP] tile (J, J) of M, upper triangle
  float* Pd = Md + T * SP;      // [T][SP] columns [I T, I T + T) of P' for this tile's rows
  float* Bk = Pd + T * SP;      // [T][SP] bulk maximum
  float* As = Bk + T * SP;      // [KT][AP] P' slice, transposed
  float* Bs = As + KT * AP;     // [KT][T] M slice
  float* Prow = Bs + KT * T;    // [T + 1] P'[i][J T .. J T + T] of the current row
  float* Pleft = Prow + T + 1;  // [T] P'[I T + r][J T]
  float* Mleft = Pleft + T;     // [T] M[I T + 1 + r][J T - 1]
  float* Mb = Mleft + T;        // [T] M[I T + T][J T + x]
  __shared__ int s_last;

  const int tid = threadIdx.x;
  const int slot = blockIdx.x / S, s = blockIdx.x - slot * S;
  int lo = 0, hi = count - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (maps[mid].ntpre - mid * delta <= slot) lo = mid;
    else hi = mid - 1;
  }
  const FoldMap mp = maps[lo];
  const int I = slot - (mp.ntpre - lo * delta), J = I + delta;
  const int ld = mp.ld, i0 = I * T, j0 = J * T;
  float* __restrict__ Mg = mp.M;
  float* __restrict__ Pg = mp.P;

  // ---- (a) bulk
  if (delta >= 2) {
    const int ty = tid / 16, tx = tid % 16;
    float acc[TM][TM];
#pragma unroll
    for (int a = 0; a < TM; ++a)
#pragma unroll
      for (int b = 0; b < TM; ++b) acc[a][b] = -INFINITY;
    const int nk = delta - 1;
    const int c_begin = (I + 1 + (int)((long long)s * nk / S)) * T;
    const int c_end = (I + 1 + (int)((long long)(s + 1) * nk / S)) * T;
    constexpr int kVec = T * KT / 4;  // float4 per operand slice
    const bool loader = tid < kVec;
    const int ar = tid / (KT / 4), aq = tid % (KT / 4);
    const int br = tid / (T / 4), bq = tid % (T / 4);
    float4 an = make_float4(0.f, 0.f, 0.f, 0.f), bn = an;
    if (loader) {
      an = *reinterpret_cast<const float4*>(Pg + (long long)(i0 + ar) * ld + c_begin + aq * 4);
      bn = *reinterpret_cast<const float4*>(Mg + (long long)(c_begin + br) * ld + j0 + bq * 4);
    }
    for (int c0 = c_begin; c0 < c_end; c0 += KT) {
      __syncthreads();
      if (loader) {
        As[(aq * 4 + 0) * AP + ar] = an.x;
        As[(aq * 4 + 1) * AP + ar] = an.y;
        As[(aq * 4 + 2) * AP + ar] = an.z;
        As[(aq * 4 + 3) * AP + ar] = an.w;
        *reinterpret_cast<float4*>(Bs + br * T + bq * 4) = bn;
      }
      __syncthreads();
      if (loader && c0 + KT < c_end) {
        an = *reinterpret_cast<const float4*>(Pg + (long long)(i0 + ar) * ld + c0 + KT + aq * 4);
        bn = *reinterpret_cast<const float4*>(Mg + (long long)(c0 + KT + br) * ld + j0 + bq * 4);
      }
#pragma unroll
      for (int kk = 0; kk < KT; ++kk) {
        float a[TM], b[TM];
        lds_vec(a, As + kk * AP + ty * TM);
        lds_vec(b, Bs + kk * T + tx * TM);
#pragma unroll
        for (int x = 0; x < TM; ++x)
#pragma unroll
          for (int y = 0; y < TM; ++y) acc[x][y] = fmaxf(acc[x][y], a[x] + b[y]);
      }
    }
    if (S == 1) {
#pragma unroll
      for (int a = 0; a < TM; ++a)
#pragma unroll
        for (int b = 0; b < TM; ++b) Bk[(ty * TM + a) * SP + tx * TM + b] = acc[a][b];
    } else {
      float* mine = partial + ((size_t)slot * S + s) * T * T;
#pragma unroll
      for (int a = 0; a < TM; ++a)
#pragma unroll
        for (int b = 0; b < TM; ++b) mine[(ty * TM + a) * T + tx * TM + b] = acc[a][b];
      __threadfence();
      __syncthreads();
      if (tid == 0) s_last = atomicAdd(&counters[slot], 1) == S - 1;
      __syncthreads();
      if (!s_last) return;
      __threadfence();
      const float* all = partial + (size_t)slot * S * T * T;
      for (int e = tid; e < T * T; e += kFoldThreads) {
        float v = -INFINITY;
        for (int q = 0; q < S; ++q) v = fmaxf(v, __ldcg(all + (size_t)q * T * T + e));
        Bk[(e / T) * SP + e % T] = v;
      }
      if (tid == 0) counters[slot] = 0;  // ready for the next diagonal
    }
  }

  // ---- operands of the in-tile part from earlier diagonals
  if (delta >= 1) {
    for (int e = tid; e < T * T; e += kFoldThreads) {
      const int r = e / T, x = e % T;
      if (r <= x) Md[r * SP + x] = Mg[(long long)(j0 + r) * ld + j0 + x];
      Pd[r * SP + x] = Pg[(long long)(i0 + r) * ld + i0 + x];
    }
  }
  if (tid < T) {
    const int r = tid;
    Mleft[r] = (i0 + 1 + r <= j0 - 1) ? Mg[(long long)(i0 + 1 + r) * ld + j0 - 1] : 0.f;
    Pleft[r] = Pg[(long long)(i0 + r) * ld + j0];
    Mb[r] = delta >= 1 ? Mg[(long long)(i0 + T) * ld + j0 + r] : 0.f;
  }
  __syncthreads();

  // ---- (b) in-tile, bottom-up
  const int xc = tid / G, part = tid % G;
  float wnext = tid < T ? Pg[(long long)(i0 + T - 1) * ld + j0 + tid + 1] : 0.f;
  for (int r = T - 1; r >= 0; --r) {
    const int i = i0 + r;
    if (tid < T) {
      const int x = tid, k = j0 + x;
      const float w = wnext;
      if (r > 0) wnext = Pg[(long long)(i - 1) * ld + k + 1];
      float p = -INFINITY;
      if (w != -INFINITY) {
        float m;
        if (k - 1 < i + 1) m = 0.f;
        else if (x == 0) m = Mleft[r];
        else if (r + 1 < T) m = Mc[(r + 1) * SP + x - 1];
        else m = Mb[x - 1];
        p = w + m;
        Pg[(long long)i * ld + k + 1] = p;
      }
      Prow[x + 1] = p;
      if (x == 0) Prow[0] = Pleft[r];
    }
    __syncthreads();
    const int j = j0 + xc;
    const bool valid = j >= i;
    float best = -INFINITY;
    if (valid) {
      if (delta >= 1) {
        for (int c = i + 2 + part; c < i0 + T; c += G) best = fmaxf(best, Pd[r * SP + c - i0] + Mc[(c - i0) * SP + xc]);
        for (int c = j0 + part; c <= j; c += G) best = fmaxf(best, Prow[c - j0] + Md[(c - j0) * SP + xc]);
      } else {
        for (int c = i + 2 + part; c <= j; c += G) best = fmaxf(best, Prow[c - j0] + Mc[(c - i0) * SP + xc]);
      }
    }
#pragma unroll
    for (int o = G / 2; o >= 1; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (valid && part == 0) {
      if (j >= i + 1) best = fmaxf(best, Prow[xc + 1] + 0.f);  // k = j: P[i][j] + M[j+1][j]
      if (delta >= 2) best = fmaxf(best, Bk[r * SP + xc]);
      const float below = i + 1 > j ? 0.f : (r + 1 < T ? Mc[(r + 1) * SP + xc] : Mb[xc]);
      const float v = fmaxf(below + mp.u[i], best);
      Mc[r * SP + xc] = v;
      Mg[(long long)i * ld + j] = v;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ traceback
static __device__ __forceinline__ int block_min(int v, int* red) {
  v = __reduce_min_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  int r = red[0];
#pragma unroll
  for (int w = 1; w < kFoldThreads / 32; ++w) r = min(r, red[w]);
  __syncthreads();
  return r;
}

// One CTA per map.  From (0, L - 1): i is unpaired if M[i][j] == M[i+1][j] + u[i] (256 rows tested at once, the
// first failure found by a min-index reduction); otherwise i pairs with the smallest k such that
// P[i][k] + M[k+1][j] == M[i][j] (min-index reduction), (k + 1, j) goes on the stack and (i + 1, k - 1) is next.
__global__ void __launch_bounds__(kFoldThreads)
fold_traceback_kernel(const FoldMap* __restrict__ maps, float* __restrict__ scores) {
  __shared__ int red[kFoldThreads / 32];
  __shared__ int s_i, s_j, s_sp;
  const FoldMap mp = maps[blockIdx.x];
  const int L = mp.L, ld = mp.ld, tid = threadIdx.x;
  const float* __restrict__ M = mp.M;
  const float* __restrict__ P = mp.P;
  const float* __restrict__ u = mp.u;
  for (int x = tid; x < L; x += kFoldThreads) mp.pairs[x] = -1;
  if (tid == 0) {
    s_i = 0, s_j = L - 1, s_sp = 0;
    scores[mp.out] = M[L - 1];
  }
  __syncthreads();
  for (;;) {
    int i = s_i;
    const int j = s_j;
    if (i <= j) {
      int first = INT_MAX;
      for (int base = i; base <= j && first == INT_MAX; base += kFoldThreads) {
        const int ip = base + tid;
        int cand = INT_MAX;
        if (ip <= j) {
          const float below = ip + 1 > j ? 0.f : M[(long long)(ip + 1) * ld + j];
          if (!(M[(long long)ip * ld + j] == below + u[ip])) cand = ip;
        }
        first = block_min(cand, red);
      }
      if (first != INT_MAX) {
        i = first;
        const float target = M[(long long)i * ld + j];
        int kbest = INT_MAX;
        for (int base = i + 1; base <= j && kbest == INT_MAX; base += kFoldThreads) {
          const int k = base + tid;
          int cand = INT_MAX;
          if (k <= j) {
            const float below = k + 1 > j ? 0.f : M[(long long)(k + 1) * ld + j];
            if (P[(long long)i * ld + k + 1] + below == target) cand = k;
          }
          kbest = block_min(cand, red);
        }
        if (tid == 0) {
          s_i = i + 1;
          // M[i][j] is one of its candidates, so kbest exists unless the tables hold NaN (the flag is set then)
          if (kbest != INT_MAX) {
            mp.pairs[i] = kbest, mp.pairs[kbest] = i;
            if (kbest + 1 <= j) {
              mp.stack[2 * s_sp] = kbest + 1, mp.stack[2 * s_sp + 1] = j;
              ++s_sp;
            }
            s_j = kbest - 1;
          }
        }
        __syncthreads();
        continue;
      }
    }
    // interval finished
    if (s_sp == 0) break;
    __syncthreads();
    if (tid == 0) {
      --s_sp;
      s_i = mp.stack[2 * s_sp], s_j = mp.stack[2 * s_sp + 1];
    }
    __syncthreads();
  }
}

template <int T>
static int fold_fill_launches(const FoldPlan& p, const FoldMap* desc, float* partial, int* counters, cudaStream_t st) {
  constexpr int smem = fold_fill_smem<T>();
  RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(fold_fill_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  for (int d = 0; d < p.ntmax; ++d) {
    int count = 0;
    for (int m : p.order) count += p.nt[m] > d;
    const int S = fold_splits(d, p.tiles[d]);
    fold_fill_kernel<T><<<(unsigned)(p.tiles[d] * S), kFoldThreads, smem, st>>>(desc, count, d, S, partial, counters);
  }
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

size_t rnamsm_fold_workspace_bytes(int n, const int* L) {
  FoldPlan p;
  if (fold_plan(n, L, p)) return 0;
  return p.total;
}

int rnamsm_fold(int n, const float* const* maps, const int* L, const uint8_t* const* seqs, int mode, double gamma,
                float threshold, int min_loop, int canonical, int* const* pairs_out, float* scores_out,
                void* workspace, size_t workspace_bytes, void* stream) {
  FoldPlan p;
  if (int rc = fold_plan(n, L, p)) return rc;
  RNAMSM_REQUIRE(maps && pairs_out && scores_out && workspace, "fold: maps, pairs_out, scores_out and workspace required");
  RNAMSM_REQUIRE(mode == RNAMSM_FOLD_MEA || mode == RNAMSM_FOLD_SCORE, "fold: mode %d is not RNAMSM_FOLD_MEA or "
                 "RNAMSM_FOLD_SCORE", mode);
  RNAMSM_REQUIRE(mode != RNAMSM_FOLD_MEA || (gamma > 0.0 && isfinite(gamma) && isfinite((float)(2.0 * gamma))),
                 "fold: gamma %g must be positive and 2 gamma finite in fp32", gamma);
  RNAMSM_REQUIRE(isfinite(threshold), "fold: threshold %g must be finite", (double)threshold);
  RNAMSM_REQUIRE(min_loop >= 0, "fold: min_loop %d must be >= 0", min_loop);
  RNAMSM_REQUIRE(!canonical || seqs, "fold: canonical pairing needs the sequences");
  for (int m = 0; m < n; ++m) {
    RNAMSM_REQUIRE(maps[m] && pairs_out[m], "fold: map %d: map and pairs_out required", m);
    RNAMSM_REQUIRE(!canonical || seqs[m], "fold: map %d: canonical pairing needs its sequence", m);
  }
  RNAMSM_REQUIRE(workspace_bytes >= p.total, "fold: workspace %zu < required %zu", workspace_bytes, p.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "fold: workspace must be 256 B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  std::vector<FoldMap> desc(n);
  int ntpre = 0;
  for (int q = 0; q < n; ++q) {
    const int m = p.order[q];
    FoldMap& d = desc[q];
    d.S = maps[m];
    d.seq = canonical ? seqs[m] : nullptr;
    d.pairs = pairs_out[m];
    d.M = reinterpret_cast<float*>(ws + p.M[m]);
    d.P = reinterpret_cast<float*>(ws + p.P[m]);
    d.u = reinterpret_cast<float*>(ws + p.u[m]);
    d.stack = reinterpret_cast<int*>(ws + p.stack[m]);
    d.L = L[m], d.nt = p.nt[m], d.Lp = p.nt[m] * p.T, d.ld = d.Lp + 4;
    d.ntpre = ntpre, d.out = m;
    ntpre += p.nt[m];
  }
  FoldMap* ddesc = reinterpret_cast<FoldMap*>(ws + p.desc);
  int* flag = reinterpret_cast<int*>(ws);
  int* counters = reinterpret_cast<int*>(ws + p.counters);
  float* partial = reinterpret_cast<float*>(ws + p.partial);
  RNAMSM_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
  RNAMSM_CHECK_CUDA(cudaMemcpyAsync(ddesc, desc.data(), (size_t)n * sizeof(FoldMap), cudaMemcpyHostToDevice, st));
  const int gx = std::min(p.nt[p.order[0]] * p.T, 148 * 8);
  const int mea = mode == RNAMSM_FOLD_MEA;
  fold_prep_kernel<<<dim3(gx, n), kFoldThreads, 0, st>>>(ddesc, mea, mea ? (float)(2.0 * gamma) : 1.f, threshold,
                                                         min_loop, canonical, flag, counters, ntpre);
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  const int rc = p.T == 32 ? fold_fill_launches<32>(p, ddesc, partial, counters, st)
                           : fold_fill_launches<64>(p, ddesc, partial, counters, st);
  if (rc) return rc;
  fold_traceback_kernel<<<n, kFoldThreads, 0, st>>>(ddesc, scores_out);
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  count_launch(p.ntmax + 2);
  return 0;
}

}  // extern "C"
