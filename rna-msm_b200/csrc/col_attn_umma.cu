// K7, 16-bit path, shallow MSAs (R <= 128): flash-style column attention on tcgen05 (modules.py:896-923).
// Deeper MSAs run the persistent warp-specialised kernel in col_attn_fa.cu.
//
// For every alignment column c and head h the MSA depth R is the sequence axis:
//   ctx[i,c,h,:] = sum_j softmax_j(q[i,c,h,:] . k[j,c,h,:]) v[j,c,h,:]          (q pre-scaled by 64^-0.5)
// The R x R probabilities are never materialised (the reference keeps [H,C,B,R,R] per layer).
//
// One CTA = one (c, h, 128-query block); 128 threads, thread t owns query row t = TMEM lane t.
// Per 64-key block:   S = Q K^T  (tcgen05.mma M128 N64 K64, fp32 in TMEM columns [0,64))
//                     online softmax in registers (exp2, running max / sum), P -> smem as the
//                     bf16 K-major SWIZZLE_128B A operand of the second MMA
//                     O_blk = P V (V read in place as an MN-major B operand, TMEM columns [64,128))
//                     o = o * corr + O_blk in registers.
// Q/K/V tiles come straight out of the packed q|k|v activation [R, C, 3D] through 3-D TMA boxes
// (64 d x 1 column x rows), K/V double-buffered so the next block's loads overlap this block's
// math.  64 KiB smem and 128 TMEM columns per CTA -> 3 CTAs per SM interleave MMA and softmax.
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

namespace {

constexpr int BQ = 128, BKV = 64, HD = 64;
constexpr int Q_BYTES = BQ * HD * 2;    // 16 KiB
constexpr int KV_BYTES = BKV * HD * 2;  // 8 KiB
constexpr int P_BYTES = BQ * BKV * 2;   // 16 KiB
constexpr int kSmem = Q_BYTES + 4 * KV_BYTES + P_BYTES + 128 + 1024;
constexpr int kTmemCols = 128;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(128)
col_attn_umma_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_kv, int R, int C,
                     int H, int fp16, int col_major, const uint8_t* __restrict__ pad, uint16_t* __restrict__ ctx) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Q_BYTES;            // 2 buffers
  uint8_t* sV = sK + 2 * KV_BYTES;       // 2 buffers
  uint8_t* sP = sV + 2 * KV_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + P_BYTES);
  uint64_t* q_full = bars;               // 1
  uint64_t* kv_full = bars + 1;          // 2
  uint64_t* s_ready = bars + 3;          // 1
  uint64_t* o_ready = bars + 4;          // 1
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c = blockIdx.x, h = blockIdx.y, i0 = blockIdx.z * BQ;
  const int D = H * HD;
  const int nblk = (R + BKV - 1) / BKV;
  const bool leader = (tid == 0);

  if (leader) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_kv);
    mbar_init(q_full, 1);
    mbar_init(&kv_full[0], 1);
    mbar_init(&kv_full[1], 1);
    mbar_init(s_ready, 1);
    mbar_init(o_ready, 1);
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
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + BKV;
  pdl_launch_dependents();
  pdl_wait();                // programmatic dependent launch: the prologue overlapped the predecessor's tail

  const uint32_t idesc_s = make_idesc_16(BQ, BKV, fp16, 0, 0);  // Q (K-major) x K (K-major)
  const uint32_t idesc_o = make_idesc_16(BQ, HD, fp16, 0, 1);   // P (K-major) x V (MN-major)

  auto load_kv = [&](int jb) {
    const int b = jb & 1;
    mbar_expect_tx(&kv_full[b], 2 * KV_BYTES);
    tma_load_3d(sK + b * KV_BYTES, &tm_kv, &kv_full[b], D + h * HD, col_major ? jb * BKV : c, col_major ? c : jb * BKV);
    tma_load_3d(sV + b * KV_BYTES, &tm_kv, &kv_full[b], 2 * D + h * HD, col_major ? jb * BKV : c,
                col_major ? c : jb * BKV);
  };
  auto issue_s = [&](int jb) {  // S = Q K_jb^T
    const int b = jb & 1;
    const uint32_t qa = smem_u32(sQ), ka = smem_u32(sK + b * KV_BYTES);
#pragma unroll
    for (int k = 0; k < HD / 16; ++k)
      umma_16(tmem_S, make_smem_desc_sw128(qa + k * 32, 16, 1024), make_smem_desc_sw128(ka + k * 32, 16, 1024),
                idesc_s, (uint32_t)(k != 0));
    umma_commit(s_ready);
  };
  auto issue_o = [&](int jb) {  // O_blk = P V_jb
    const int b = jb & 1;
    const uint32_t pa = smem_u32(sP), va = smem_u32(sV + b * KV_BYTES);
#pragma unroll
    for (int k = 0; k < BKV / 16; ++k)
      umma_16(tmem_O, make_smem_desc_sw128(pa + k * 32, 16, 1024),
                make_smem_desc_sw128(va + k * 2048, 8192, 1024), idesc_o, (uint32_t)(k != 0));
    umma_commit(o_ready);
  };

  if (leader) {
    mbar_expect_tx(q_full, Q_BYTES);
    tma_load_3d(sQ, &tm_q, q_full, h * HD, col_major ? i0 : c, col_major ? c : i0);
    load_kv(0);
    if (nblk > 1) load_kv(1);
    mbar_wait(q_full, 0);
    mbar_wait(&kv_full[0], 0);
    tc_fence_after();
    issue_s(0);
  }
  __syncwarp();

  const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
  const int row = tid;  // query row inside the block == TMEM lane
  constexpr float kLog2e = 1.4426950408889634f;
  float m_run = -INFINITY, l_run = 0.f;
  float o[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) o[d] = 0.f;

  for (int jb = 0; jb < nblk; ++jb) {
    const int j0 = jb * BKV;
    // key mask bits for this block: bit j set => logit forced to -10000 (padded key)
    uint32_t mask_lo = 0, mask_hi = 0;
    if (pad != nullptr) {
      const int ja = j0 + lane, jb2 = j0 + 32 + lane;
      mask_lo = __ballot_sync(0xffffffffu, ja < R && pad[(size_t)ja * C + c] != 0);
      mask_hi = __ballot_sync(0xffffffffu, jb2 < R && pad[(size_t)jb2 * C + c] != 0);
    }
    const int n_valid = min(BKV, R - j0);

    mbar_wait(s_ready, jb & 1);
    tc_fence_after();
    uint32_t sv[2][32];
    tmem_ld_32x32(tmem_S + lane_off, sv[0]);
    tmem_ld_32x32(tmem_S + lane_off + 32, sv[1]);
    tmem_ld_wait();

    float s[BKV];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < BKV; ++j) {
      float v = __uint_as_float(sv[j >> 5][j & 31]);
      const uint32_t mbits = (j < 32) ? mask_lo : mask_hi;
      if ((mbits >> (j & 31)) & 1u) v = -10000.f;  // masked_fill, modules.py:911-915
      if (j >= n_valid) v = -INFINITY;             // key row does not exist
      s[j] = v;
      mx = fmaxf(mx, v);
    }
    const float m_new = fmaxf(m_run, mx);          // finite: block has >= 1 existing key
    const float corr = ex2((m_run - m_new) * kLog2e);
    const float mscaled = m_new * kLog2e;
    float psum = 0.f;
    uint32_t pk[BKV / 2];
#pragma unroll
    for (int j = 0; j < BKV; j += 2) {
      const float p0 = ex2(fmaf(s[j], kLog2e, -mscaled));
      const float p1 = ex2(fmaf(s[j + 1], kLog2e, -mscaled));
      psum += p0 + p1;
      pk[j >> 1] = fp16 ? pack_f16(p0, p1) : pack_bf16(p0, p1);
    }
    l_run = l_run * corr + psum;
    m_run = m_new;
    // P row -> smem, K-major SWIZZLE_128B: 16-byte chunk ch of row r lives at chunk (ch ^ (r & 7)).
    {
      uint8_t* prow = sP + row * 128;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        const uint4 val = make_uint4(pk[ch * 4], pk[ch * 4 + 1], pk[ch * 4 + 2], pk[ch * 4 + 3]);
        *reinterpret_cast<uint4*>(prow + ((ch ^ (row & 7)) << 4)) = val;
      }
    }
    tc_fence_before();          // our tcgen05.ld of S precede the barrier (S is overwritten next)
    fence_proxy_async_smem();   // generic-proxy P writes -> visible to the tensor-core (async) proxy
    __syncthreads();
    if (leader) {
      tc_fence_after();
      issue_o(jb);
      if (jb + 1 < nblk) {
        mbar_wait(&kv_full[(jb + 1) & 1], ((jb + 1) >> 1) & 1);
        tc_fence_after();
        issue_s(jb + 1);
      }
    }
    __syncwarp();
    mbar_wait(o_ready, jb & 1);
    tc_fence_after();
    if (leader && jb + 2 < nblk) load_kv(jb + 2);  // buffer (jb & 1) is free: S(jb) and O(jb) are done
    __syncwarp();
    uint32_t ov[2][32];
    tmem_ld_32x32(tmem_O + lane_off, ov[0]);
    tmem_ld_32x32(tmem_O + lane_off + 32, ov[1]);
    tmem_ld_wait();
#pragma unroll
    for (int d = 0; d < HD; ++d) o[d] = fmaf(o[d], corr, __uint_as_float(ov[d >> 5][d & 31]));
    tc_fence_before();          // O loads precede the next block's barrier / PV MMA
  }

  const int i = i0 + row;
  if (i < R) {
    const float inv = 1.f / l_run;
    uint16_t* dst = ctx + ((size_t)i * C + c) * D + h * HD;
#pragma unroll
    for (int d = 0; d < HD; d += 8) {
      uint4 val;
      if (fp16)
        val = make_uint4(pack_f16(o[d] * inv, o[d + 1] * inv), pack_f16(o[d + 2] * inv, o[d + 3] * inv),
                         pack_f16(o[d + 4] * inv, o[d + 5] * inv), pack_f16(o[d + 6] * inv, o[d + 7] * inv));
      else
        val = make_uint4(pack_bf16(o[d] * inv, o[d + 1] * inv), pack_bf16(o[d + 2] * inv, o[d + 3] * inv),
                         pack_bf16(o[d + 4] * inv, o[d + 5] * inv), pack_bf16(o[d + 6] * inv, o[d + 7] * inv));
      *reinterpret_cast<uint4*>(dst + d) = val;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

int launch_col_attn_small_16(const void* qkv, int R, int C, int H, int fp16, int col_major, const uint8_t* pad, void* ctx,
                             cudaStream_t st) {
  RNAMSM_REQUIRE(R >= 1 && C >= 1 && H >= 1 && C <= 2147483647 / 1 && H <= 65535, "col_attn_bf16: bad shape");
  const int ld = 3 * H * HD;
  CUtensorMap tq, tkv;
  uint64_t dims[3] = {(uint64_t)ld, (uint64_t)(col_major ? R : C), (uint64_t)(col_major ? C : R)};
  uint64_t strides[2] = {(uint64_t)ld * 2, (uint64_t)(col_major ? R : C) * ld * 2};
  uint32_t box_q[3] = {HD, (uint32_t)(col_major ? BQ : 1), (uint32_t)(col_major ? 1 : BQ)};
  uint32_t box_kv[3] = {HD, (uint32_t)(col_major ? BKV : 1), (uint32_t)(col_major ? 1 : BKV)};
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  if (encode_tmap(&tq, in_dt, qkv, 3, dims, strides, box_q)) return 3;
  if (encode_tmap(&tkv, in_dt, qkv, 3, dims, strides, box_kv)) return 3;
  RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(col_attn_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
  dim3 grid(C, H, ceil_div(R, BQ));
  RNAMSM_REQUIRE(grid.z <= 65535, "col_attn_bf16: R too large");
  ProfScope prof(KC_COL_ATTN, st);
  RNAMSM_CHECK_CUDA(launch_pdl(col_attn_umma_kernel, grid, dim3(128), kSmem, st, tq, tkv, R, C, H, fp16, col_major, pad,
                               reinterpret_cast<uint16_t*>(ctx)));
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int launch_col_attn_fa_16(const void* qkv, int R, int C, int H, int fp16, int col_major, const uint8_t* pad, void* ctx,
                          cudaStream_t st);   // col_attn_fa.cu

// Dispatch: MSAs deeper than one 128-row query tile run the persistent warp-specialised kernel
// (col_attn_fa.cu: two query tiles per work item); shallow ones (R <= 128) keep this
// one-tile-per-CTA kernel, whose single tile wastes nothing.
int launch_col_attn_16(const void* qkv, int R, int C, int H, int fp16, int col_major, const uint8_t* pad, void* ctx,
                       cudaStream_t st) {
  if (R <= 128) return launch_col_attn_small_16(qkv, R, C, H, fp16, col_major, pad, ctx, st);
  return launch_col_attn_fa_16(qkv, R, C, H, fp16, col_major, pad, ctx, st);
}

}  // namespace rnamsm
