// Column-attention probabilities on request (modules.py:907-918, the [H, C, B, R, R] tensor the reference returns):
//   s_ij          = q[i,c,h,:] . k[j,c,h,:]          (q pre-scaled by 64^-0.5 in the QKV epilogue)
//                   replaced by -10000 where key j of column c is padded (masked_fill, modules.py:911-915)
//   P[h, c, i, j] = softmax_j(s_ij)
//   mean[h, i, j] = (1/C) sum_c P[h, c, i, j]        (without the full tensor existing anywhere)
// The flash kernels (col_attn_umma.cu, col_attn_fa.cu, simt_f32.cu) never form P, so these read the
// same q|k buffer and pad flags again, in two passes:
//   1. lse: one CTA per (column, head, query tile) streams the key blocks of its column and keeps a running max / sum;
//      the row's max m[h, c, i] and log-sum log(sum_j exp(s_ij - m)) go to two fp32 [H, C, R] scratch arrays.  They stay
//      apart because a fully padded column has m = -10000, where one fp32 ulp is 1e-3: m + log(R) rounded to fp32 would
//      put a 5e-4 relative error on its uniform probabilities, (s - m) - log(sum) is exact there.
//   2. probs: one CTA per (head, query tile, key tile) loops over the C columns, forms P = exp((s - m) - log(sum)), stores the
//      tile (full form) and / or adds it into registers (mean).  The column sum runs in column order inside one CTA:
//      deterministic, no atomics, one kernel for both outputs.
// 16-bit path: S = Q K^T on tcgen05 (M128 N128 K64, fp32 in tensor memory), operands by TMA in either q|k layout;
// exponentials in base 2 (ex2.approx), max and log-sum stored in base 2.  fp32 path: FFMA tiles, expf / logf.
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

namespace {

constexpr int BT = 128, HD = 64;
constexpr int TILE_BYTES = BT * HD * 2;      // 16 KiB: 128 rows x 64 dims, 16-bit, SWIZZLE_128B
constexpr int STAGE_BYTES = 2 * TILE_BYTES;  // Q tile | K tile
constexpr int STG_LD = 33;                   // per-warp 32 x 32 fp32 transpose buffer, padded against bank conflicts
constexpr int STG_BYTES = 4 * 32 * STG_LD * 4;
constexpr int kSmem = 2 * STAGE_BYTES + STG_BYTES + 64 + 1024;
constexpr int kTmemCols = 2 * BT;            // S double-buffered: MMA of step s+1 overlaps the exponentials of step s
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// kMode 0: pass 1 (lse).  Otherwise pass 2: bit 0 = store P, bit 1 = accumulate the column mean.
// Pass 1: blockIdx = (c, h, query tile), step s = key block s.  Pass 2: blockIdx = (key tile, query tile, h), step s =
// column s.  128 threads; thread t owns query row i0 + t = TMEM lane t.
template <int kMode>
__global__ void __launch_bounds__(128)
col_probs_umma_kernel(const __grid_constant__ CUtensorMap tm, int R, int C, int H, int fp16, int col_major,
                      const uint8_t* __restrict__ pad, float* __restrict__ lse2, float* __restrict__ probs,
                      float* __restrict__ mean) {
  constexpr bool kFull = (kMode & 1) != 0, kMean = (kMode & 2) != 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* stage = smem;                                                    // 2 stages
  float* stg = reinterpret_cast<float*>(smem + 2 * STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * STAGE_BYTES + STG_BYTES);
  uint64_t* full = bars;       // 2
  uint64_t* s_ready = bars + 2;  // 2
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = H * HD;
  const int h = kMode == 0 ? blockIdx.y : blockIdx.z;
  const int i0 = (kMode == 0 ? blockIdx.z : blockIdx.y) * BT;
  const int nsteps = kMode == 0 ? (R + BT - 1) / BT : C;
  auto step_col = [&](int s) { return kMode == 0 ? (int)blockIdx.x : s; };
  auto step_j0 = [&](int s) { return kMode == 0 ? s * BT : (int)blockIdx.x * BT; };

  if (tid == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    mbar_init(&s_ready[0], 1);
    mbar_init(&s_ready[1], 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t idesc = make_idesc_16(BT, BT, fp16, 0, 0);   // Q (K-major) x K (K-major)

  auto load = [&](int s) {
    uint8_t* sq = stage + (s & 1) * STAGE_BYTES;
    const int c = step_col(s), j0 = step_j0(s);
    const bool need_q = kMode != 0 || s < 2;   // pass 1: the query tile stays put, both stages keep their copy
    mbar_expect_tx(&full[s & 1], need_q ? STAGE_BYTES : TILE_BYTES);
    if (need_q) tma_load_3d(sq, &tm, &full[s & 1], h * HD, col_major ? i0 : c, col_major ? c : i0);
    tma_load_3d(sq + TILE_BYTES, &tm, &full[s & 1], D + h * HD, col_major ? j0 : c, col_major ? c : j0);
  };
  auto issue = [&](int s) {
    const uint32_t qa = smem_u32(stage + (s & 1) * STAGE_BYTES), ka = qa + TILE_BYTES;
#pragma unroll
    for (int k = 0; k < HD / 16; ++k)
      umma_16(tmem_base + (s & 1) * BT, make_smem_desc_sw128(qa + k * 32, 16, 1024),
              make_smem_desc_sw128(ka + k * 32, 16, 1024), idesc, (uint32_t)(k != 0));
    umma_commit(&s_ready[s & 1]);
  };

  if (tid == 0) {
    load(0);
    if (nsteps > 1) load(1);
    mbar_wait(&full[0], 0);
    tc_fence_after();
    issue(0);
  }
  __syncwarp();

  const int i = i0 + tid;
  const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
  float* st = stg + warp * 32 * STG_LD;
  float m2 = -INFINITY, l = 0.f;                 // pass 1: running max (base 2) and sum
  float acc[kMean ? BT : 1];
#pragma unroll
  for (int k = 0; k < (kMean ? BT : 1); ++k) acc[k] = 0.f;

  for (int s = 0; s < nsteps; ++s) {
    const int c = step_col(s), j0 = step_j0(s);
    const size_t row_idx = ((size_t)h * C + c) * R + i;
    const float my_max = (kMode != 0 && i < R) ? lse2[row_idx] : 0.f;
    const float my_lsum = (kMode != 0 && i < R) ? lse2[(size_t)H * C * R + row_idx] : 0.f;
    if (tid == 0 && s + 1 < nsteps) {
      mbar_wait(&full[(s + 1) & 1], ((s + 1) >> 1) & 1);
      tc_fence_after();
      issue(s + 1);
    }
    __syncwarp();
    mbar_wait(&s_ready[s & 1], (s >> 1) & 1);
    tc_fence_after();
    if (tid == 0 && s + 2 < nsteps) load(s + 2);   // MMA(s) has finished reading its stage
    __syncwarp();
    const uint32_t tS = tmem_base + (s & 1) * BT + lane_off;
#pragma unroll
    for (int jc = 0; jc < BT / 32; ++jc) {
      const int jl = j0 + jc * 32 + lane;
      const uint32_t mbits = pad ? __ballot_sync(0xffffffffu, jl < R && pad[(size_t)jl * C + c] != 0) : 0u;
      const int n_valid = R - (j0 + jc * 32);     // key j0 + jc*32 + k exists for k < n_valid
      uint32_t sv[32];
      tmem_ld_32x32(tS + jc * 32, sv);
      tmem_ld_wait();
      if (kMode == 0) {
        float s2[32];
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          float v = __uint_as_float(sv[k]);
          if ((mbits >> k) & 1u) v = -10000.f;
          s2[k] = k < n_valid ? __fmul_rn(v, kLog2e) : -INFINITY;   // no FMA contraction: pass 2 rounds s2 alike
          mx = fmaxf(mx, s2[k]);
        }
        if (mx > -INFINITY) {
          const float mn = fmaxf(m2, mx);
          float sum = 0.f;
#pragma unroll
          for (int k = 0; k < 32; ++k) sum += ex2(s2[k] - mn);
          l = l * ex2(m2 - mn) + sum;
          m2 = mn;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          float v = __uint_as_float(sv[k]);
          if ((mbits >> k) & 1u) v = -10000.f;
          const float p = ex2((__fmul_rn(v, kLog2e) - my_max) - my_lsum);
          if (kMean) acc[jc * 32 + k] += p;
          if (kFull) st[lane * STG_LD + k] = p;
        }
        if (kFull) {   // transpose through shared memory: each store instruction writes 32 consecutive keys of one row
          __syncwarp();
          if (jl < R) {
            float* dst = probs + (((size_t)h * C + c) * R + i0 + warp * 32) * R + jl;
            const int rows = min(32, R - (i0 + warp * 32));
            for (int r = 0; r < rows; ++r) __stcs(dst + (size_t)r * R, st[r * STG_LD + lane]);
          }
          __syncwarp();
        }
      }
    }
    tc_fence_before();
    __syncthreads();   // TMEM buffer (s & 1) fully read before MMA(s + 2) overwrites it
  }

  if (kMode == 0) {
    if (i < R) {
      lse2[((size_t)h * C + blockIdx.x) * R + i] = m2;
      lse2[(size_t)H * C * R + ((size_t)h * C + blockIdx.x) * R + i] = log2f(l);
    }
  } else if (kMean) {
    const float fc = (float)C;
    const int j0 = blockIdx.x * BT;
#pragma unroll
    for (int jc = 0; jc < BT / 32; ++jc) {
#pragma unroll
      for (int k = 0; k < 32; ++k) st[lane * STG_LD + k] = acc[jc * 32 + k] / fc;
      __syncwarp();
      const int jl = j0 + jc * 32 + lane;
      if (jl < R) {
        float* dst = mean + ((size_t)h * R + i0 + warp * 32) * R + jl;
        const int rows = min(32, R - (i0 + warp * 32));
        for (int r = 0; r < rows; ++r) dst[(size_t)r * R] = st[r * STG_LD + lane];
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ---- fp32 path: 64 x 64 FFMA tiles, 256 threads as 16 x 16; thread (ty, tx) owns rows ty*4.. and keys tx*4.. ------
constexpr int FT = 64;

// s[a][b] = q[i0 + ty*4 + a] . k[j0 + tx*4 + b] from the tiles in shared memory ([d][row] layout)
__device__ __forceinline__ void f32_scores(const float (*Qs)[FT + 4], const float (*Ks)[FT + 4], int ty, int tx,
                                           float (&s)[4][4]) {
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) s[a][b] = 0.f;
#pragma unroll 8
  for (int d = 0; d < HD; ++d) {
    const float4 qa = *reinterpret_cast<const float4*>(&Qs[d][ty * 4]);
    const float4 kb = *reinterpret_cast<const float4*>(&Ks[d][tx * 4]);
    const float q[4] = {qa.x, qa.y, qa.z, qa.w}, k[4] = {kb.x, kb.y, kb.z, kb.w};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) s[a][b] = fmaf(q[a], k[b], s[a][b]);
  }
}

// rows r0.. of column c, head h, part (0 = q, 1 = k) -> T[d][r]; rows past R read as zero
__device__ __forceinline__ void f32_load_tile(float (*T)[FT + 4], const float* qkv, int R, int C, int H, int c, int h,
                                              int part, int r0) {
  const int ld = 3 * H * HD;
  for (int idx = threadIdx.x; idx < FT * HD; idx += 256) {
    const int d = idx & 63, r = idx >> 6;
    T[d][r] = (r0 + r < R) ? qkv[((size_t)(r0 + r) * C + c) * ld + part * H * HD + h * HD + d] : 0.f;
  }
}

__global__ void __launch_bounds__(256)
col_lse_f32_kernel(const float* __restrict__ qkv, int R, int C, int H, const uint8_t* __restrict__ pad,
                   float* __restrict__ lse) {
  __shared__ __align__(16) float Qs[HD][FT + 4];
  __shared__ __align__(16) float Ks[HD][FT + 4];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int c = blockIdx.x, h = blockIdx.y, i0 = blockIdx.z * FT;
  f32_load_tile(Qs, qkv, R, C, H, c, h, 0, i0);
  float m[4], l[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) { m[a] = -INFINITY; l[a] = 0.f; }
  for (int j0 = 0; j0 < R; j0 += FT) {
    __syncthreads();
    f32_load_tile(Ks, qkv, R, C, H, c, h, 1, j0);
    __syncthreads();
    float s[4][4];
    f32_scores(Qs, Ks, ty, tx, s);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int j = j0 + tx * 4 + b;
      const bool masked = j < R && pad && pad[(size_t)j * C + c];
#pragma unroll
      for (int a = 0; a < 4; ++a) s[a][b] = j >= R ? -INFINITY : (masked ? -10000.f : s[a][b]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      float mx = fmaxf(fmaxf(s[a][0], s[a][1]), fmaxf(s[a][2], s[a][3]));
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float mn = fmaxf(m[a], mx);   // finite: every key tile holds >= 1 existing key
      float ps = 0.f;
#pragma unroll
      for (int b = 0; b < 4; ++b) ps += expf(s[a][b] - mn);
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) ps += __shfl_xor_sync(0xffffffffu, ps, off);
      l[a] = l[a] * expf(m[a] - mn) + ps;
      m[a] = mn;
    }
  }
  if (tx == 0) {
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int i = i0 + ty * 4 + a;
      if (i < R) {
        lse[((size_t)h * C + c) * R + i] = m[a];
        lse[(size_t)H * C * R + ((size_t)h * C + c) * R + i] = logf(l[a]);
      }
    }
  }
}

__global__ void __launch_bounds__(256)
col_probs_f32_kernel(const float* __restrict__ qkv, int R, int C, int H, const uint8_t* __restrict__ pad,
                     const float* __restrict__ lse, float* __restrict__ probs, float* __restrict__ mean) {
  __shared__ __align__(16) float Qs[HD][FT + 4];
  __shared__ __align__(16) float Ks[HD][FT + 4];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int j0 = blockIdx.x * FT, i0 = blockIdx.y * FT, h = blockIdx.z;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  for (int c = 0; c < C; ++c) {
    __syncthreads();
    f32_load_tile(Qs, qkv, R, C, H, c, h, 0, i0);
    f32_load_tile(Ks, qkv, R, C, H, c, h, 1, j0);
    __syncthreads();
    float s[4][4];
    f32_scores(Qs, Ks, ty, tx, s);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int i = i0 + ty * 4 + a;
      if (i >= R) continue;
      const float mi = lse[((size_t)h * C + c) * R + i], li = lse[(size_t)H * C * R + ((size_t)h * C + c) * R + i];
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int j = j0 + tx * 4 + b;
        if (j >= R) continue;
        const float v = (pad && pad[(size_t)j * C + c]) ? -10000.f : s[a][b];
        const float p = expf((v - mi) - li);
        acc[a][b] += p;
        if (probs) __stcs(&probs[(((size_t)h * C + c) * R + i) * R + j], p);
      }
    }
  }
  if (mean) {
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int i = i0 + ty * 4 + a;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int j = j0 + tx * 4 + b;
        if (i < R && j < R) mean[((size_t)h * R + i) * R + j] = acc[a][b] / (float)C;
      }
    }
  }
}

__global__ void fill_ones_kernel(float* __restrict__ p, long long n) {
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x)
    p[k] = 1.f;
}

int fill_ones(float* p, long long n, cudaStream_t st) {
  if (p == nullptr || n <= 0) return 0;
  fill_ones_kernel<<<ceil_div(n, 256) < 1024 ? ceil_div(n, 256) : 1024, 256, 0, st>>>(p, n);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

template <int kMode>
int launch_umma(dim3 grid, cudaStream_t st, const CUtensorMap& tm, int R, int C, int H, int fp16, int col_major,
                const uint8_t* pad, float* lse2, float* probs, float* mean) {
  static bool attr_set = false;
  if (!attr_set) {
    RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(col_probs_umma_kernel<kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    attr_set = true;
  }
  col_probs_umma_kernel<kMode><<<grid, 128, kSmem, st>>>(tm, R, C, H, fp16, col_major, pad, lse2, probs, mean);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

size_t col_probs_scratch_bytes(int R, int C, int H) {
  if (R <= 0 || C <= 0 || H <= 0) return 0;
  return ((size_t)2 * H * C * R * 4 + 255) & ~(size_t)255;
}

int launch_col_probs(const void* qkv, int R, int C, int H, int dtype, int col_major, const uint8_t* pad, float* probs,
                     float* mean, void* scratch, cudaStream_t st) {
  RNAMSM_REQUIRE(R >= 1 && C >= 1 && H >= 1 && H <= 65535, "col_attn_probs: bad shape R=%d C=%d H=%d", R, C, H);
  if (probs == nullptr && mean == nullptr) return 0;
  int rc;
  if (R == 1) {   // softmax over one key: all ones (modules.py:882-894 returns torch.ones)
    if ((rc = fill_ones(probs, (long long)H * C, st)) || (rc = fill_ones(mean, H, st))) return rc;
    return 0;
  }
  RNAMSM_REQUIRE(scratch != nullptr, "col_attn_probs: scratch of rnamsm_col_probs_scratch_bytes(R, C, H) bytes required");
  RNAMSM_REQUIRE(!col_major || dtype == RNAMSM_BF16 || dtype == RNAMSM_F16,
                 "col_attn_probs: the column-major q|k|v layout exists in the 16-bit path only");
  float* lse = reinterpret_cast<float*>(scratch);
  ProfScope prof(KC_COL_ATTN, st);
  if (dtype == RNAMSM_F32) {
    dim3 g1(C, H, ceil_div(R, FT));
    dim3 g2(ceil_div(R, FT), ceil_div(R, FT), H);
    RNAMSM_REQUIRE(g1.z <= 65535, "col_attn_probs: R=%d too large", R);
    col_lse_f32_kernel<<<g1, 256, 0, st>>>((const float*)qkv, R, C, H, pad, lse);
    count_launch();
    RNAMSM_CHECK_CUDA(cudaGetLastError());
    col_probs_f32_kernel<<<g2, 256, 0, st>>>((const float*)qkv, R, C, H, pad, lse, probs, mean);
    count_launch();
    RNAMSM_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  RNAMSM_REQUIRE(dtype == RNAMSM_BF16 || dtype == RNAMSM_F16, "col_attn_probs: unknown dtype %d", dtype);
  const int ld = 3 * H * HD;
  CUtensorMap tm;
  uint64_t dims[3] = {(uint64_t)ld, (uint64_t)(col_major ? R : C), (uint64_t)(col_major ? C : R)};
  uint64_t strides[2] = {(uint64_t)ld * 2, (uint64_t)(col_major ? R : C) * ld * 2};
  uint32_t box[3] = {HD, (uint32_t)(col_major ? BT : 1), (uint32_t)(col_major ? 1 : BT)};
  const int fp16 = dtype == RNAMSM_F16;
  if (encode_tmap(&tm, fp16 ? TMAP_F16 : TMAP_BF16, qkv, 3, dims, strides, box)) return 3;
  dim3 g1(C, H, ceil_div(R, BT));
  dim3 g2(ceil_div(R, BT), ceil_div(R, BT), H);
  RNAMSM_REQUIRE(g1.z <= 65535, "col_attn_probs: R=%d too large", R);
  if ((rc = launch_umma<0>(g1, st, tm, R, C, H, fp16, col_major, pad, lse, nullptr, nullptr))) return rc;
  if (probs && mean) return launch_umma<3>(g2, st, tm, R, C, H, fp16, col_major, pad, lse, probs, mean);
  if (probs) return launch_umma<1>(g2, st, tm, R, C, H, fp16, col_major, pad, lse, probs, nullptr);
  return launch_umma<2>(g2, st, tm, R, C, H, fp16, col_major, pad, lse, nullptr, mean);
}

}  // namespace rnamsm
