// K7, 16-bit path, MSAs deeper than 128 rows: column attention with 128-key steps and P in tensor memory
// (modules.py:896-923).  For every alignment column c and head h the MSA depth R is the sequence axis:
//   ctx[i,c,h,:] = sum_j softmax_j(q[i,c,h,:] . k[j,c,h,:]) v[j,c,h,:]     (q pre-scaled by 64^-1/2)
//
// Why this shape (tools/micro/mma_chain_bench.cu, tools/micro/tmem_umma_bench.cu on a B200; DESIGN.md 4.2): the
// round-1 kernel, four query tiles with 64-key steps and P through shared memory, was held at ~3000 cycles per step
// by three resources at once --
//   shared-memory port: an M128 N64 K16 MMA with both operands in shared memory reads 6 KiB for 32 cycles of math =
//     48 cycles (measured: 4 issuing threads, 1536 cycles per 32 instructions), + 64 KiB of P stores per step
//     = ~2200 cycles;  XU: 64 ex2 x 16 warps at 16/clk/SM = 2048 cycles;  issue slots of the softmax warps: ~2400
//     cycles (the step body with every barrier satisfied, 4 warps per scheduler).
// Here a step covers 128 keys of 2 query tiles:
//   S = Q K^T as M128 N128 K16 (8 KiB per 64 cycles of math: exactly the shared-memory rate),
//   P goes registers -> TENSOR MEMORY (tcgen05.st) and P V takes its A operand from there ([a_tmem]): only V is read
//   from shared memory (2 KiB per 32-cycle instruction), no P stores, no generic->async proxy fence per step,
//   one thread = one query row with 128 logits per step, so the per-step barrier / fence / wait overhead is paid
//   once per 128 exponentials instead of once per 64, with 8 softmax warps of 216 registers instead of 16 of 96.
// That leaves the XU as the only resource near its limit (shared memory ~1000, issue ~1100 of ~2200 cycles per step).
//
// TMEM (512 columns): tile t owns columns [256 t, 256 t + 256):  S 128 | P 64 (128 keys, two per column) | O 64.
// S(g+1) is issued as soon as the softmax warps hold S(g) in registers (one step ahead); P has its own columns, so it
// does not collide with that.
//
//   warp 0 lane 0     TMA producer: Q tiles (double-buffered across items) and a K/V ring of 128-key stages
//   warps 1, 2        S issuer of tile 0 / 1 (lane 0); warp 1 owns the TMEM allocation
//   warps 4, 5        PV issuer of tile 0 / 1 (lane 0); warps 3, 6, 7 idle (roles come in whole warpgroups for setmaxnreg)
//   warps 8..15       softmax, one warpgroup per tile (thread = query row = TMEM lane): lazy rescaling (threshold 2^8),
//                     packed fp32 pair arithmetic
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

namespace {

constexpr int NT = 2, BQ = 128, BKV = 128, HD = 64;
constexpr int Q_BYTES = BQ * HD * 2;        // 16 KiB per tile
constexpr int KV_BYTES = BKV * HD * 2;      // 16 KiB each for K and V
constexpr int STG_BYTES = BQ * HD * 2;      // 16 KiB per tile: O rows staged for the TMA store
constexpr int kKvStages = 4;
constexpr int OFF_Q = 0;                                     // [2 item buffers][NT tiles]
constexpr int OFF_KV = OFF_Q + 2 * NT * Q_BYTES;             // [stages][K | V]
constexpr int OFF_STG = OFF_KV + kKvStages * 2 * KV_BYTES;   // [NT tiles]
constexpr int OFF_BAR = OFF_STG + NT * STG_BYTES;
constexpr int kSmem = OFF_BAR + 512 + 1024;
constexpr int kRoleWarps = 8;                                // two warpgroups of single-thread roles (3 warps idle)
constexpr int kThreads = 512;                                // the role warps + one softmax warpgroup per tile
constexpr int kRoleRegs = 40, kSoftmaxRegs = 216;            // setmaxnreg: 256 x 40 + 256 x 216 = 65536 = launch 512 x 128
constexpr int kTmemCols = 512;
constexpr int TM_S = 0, TM_P = 128, TM_O = 192, TM_TILE = 256;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kRescaleThreshold = 8.0f;   // log2 units: P stays <= 2^8
static_assert(kSmem <= 227 * 1024, "column attention: shared memory budget");

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Orders a volatile asm (a barrier probe) behind the computation of v without emitting an instruction.
__device__ __forceinline__ void anchor_after(float v) { asm volatile("" ::"f"(v) : "memory"); }

struct Item { int c, h, i0; };

__device__ __forceinline__ Item decode_item(int item, int nqb, int H) {
  Item it;
  it.i0 = (item % nqb) * (NT * BQ);
  item /= nqb;
  it.h = item % H;
  it.c = item / H;
  return it;
}

template <bool kFp16>
__global__ void __launch_bounds__(kThreads, 1)
col_attn_fa_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_kv,
                   const __grid_constant__ CUtensorMap tm_o, int R, int C, int H, int col_major, int n_items,
                   const uint8_t* __restrict__ pad) {
  constexpr int fp16 = kFp16 ? 1 : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* q_full = bars;                      // [2]
  uint64_t* q_empty = bars + 2;                 // [2]
  uint64_t* kv_full = bars + 4;                 // [4]
  uint64_t* kv_empty = bars + 8;                // [4]
  uint64_t* s_full = bars + 12;                 // [2] per tile
  uint64_t* s_free = bars + 14;
  uint64_t* p_full = bars + 16;
  uint64_t* pv_done = bars + 18;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 20);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int D = H * HD;
  const int nblk = (R + BKV - 1) / BKV;
  const int nqb = (R + NT * BQ - 1) / (NT * BQ);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_kv);
    tma_prefetch_desc(&tm_o);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&q_full[b], 1);
      mbar_init(&q_empty[b], NT);               // one commit per MMA issuer
      mbar_init(&s_full[b], 1);
      mbar_init(&s_free[b], 4);
      mbar_init(&p_full[b], 4);
      mbar_init(&pv_done[b], 1);
    }
    for (int b = 0; b < 4; ++b) {
      mbar_init(&kv_full[b], 1);
      mbar_init(&kv_empty[b], NT);
    }
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
  pdl_launch_dependents();
  pdl_wait();

  if (warp < kRoleWarps) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRoleRegs));
  if (warp == 0 && lane == 0) {
    // ================================ TMA producer ================================
    int kv_stage = 0;
    uint32_t kv_phase = 0;
    int li = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++li) {
      const Item it = decode_item(item, nqb, H);
      const int qb = li & 1, quse = li >> 1;
      mbar_wait_relaxed(&q_empty[qb], (quse & 1) ^ 1);
      mbar_expect_tx(&q_full[qb], NT * Q_BYTES);
#pragma unroll
      for (int t = 0; t < NT; ++t)
        tma_load_3d(smem + OFF_Q + (qb * NT + t) * Q_BYTES, &tm_q, &q_full[qb], it.h * HD,
                    col_major ? it.i0 + t * BQ : it.c, col_major ? it.c : it.i0 + t * BQ);
      for (int j = 0; j < nblk; ++j) {
        mbar_wait_relaxed(&kv_empty[kv_stage], kv_phase ^ 1);
        uint8_t* sk = smem + OFF_KV + kv_stage * 2 * KV_BYTES;
        mbar_expect_tx(&kv_full[kv_stage], 2 * KV_BYTES);
        tma_load_3d(sk, &tm_kv, &kv_full[kv_stage], D + it.h * HD, col_major ? j * BKV : it.c, col_major ? it.c : j * BKV);
        tma_load_3d(sk + KV_BYTES, &tm_kv, &kv_full[kv_stage], 2 * D + it.h * HD, col_major ? j * BKV : it.c,
                    col_major ? it.c : j * BKV);
        if (++kv_stage == kKvStages) { kv_stage = 0; kv_phase ^= 1; }
      }
    }
  } else if ((warp == 1 || warp == 2) && lane == 0) {
    // ================================ S issuer of tile t ===========================
    // S and PV have separate issuing threads: one thread doing both (12 instructions per step, each behind ~15 scalar
    // instructions of descriptor arithmetic and the barrier round trips) was the slowest stage of the pipeline -- ncu:
    // 46 % of the steps found S not ready, and with S moved ahead of PV the wait moved to PV.
    const int t = warp - 1;
    const uint32_t idesc_s = make_idesc_16(BQ, BKV, fp16, 0, 0);  // Q (K-major, smem) x K (K-major, smem), N = 128 keys
    const int my_items = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const uint32_t tmem_S = tmem_base + t * TM_TILE + TM_S;
    int s_stage = 0;
    uint32_t s_phase = 0;
    long long gs = 0;
    for (int li = 0; li < my_items; ++li) {
      const int qb = li & 1, quse = li >> 1;
      mbar_wait_relaxed(&q_full[qb], quse & 1);
      const uint32_t qa = smem_u32(smem + OFF_Q + (qb * NT + t) * Q_BYTES);
      for (int j = 0; j < nblk; ++j, ++gs) {
        mbar_wait_relaxed(&kv_full[s_stage], s_phase);
        if (gs > 0) mbar_wait_quiet(&s_free[t], (uint32_t)((gs - 1) & 1));   // softmax t holds S(gs-1) in registers
        tc_fence_after();
        const uint32_t ka = smem_u32(smem + OFF_KV + s_stage * 2 * KV_BYTES);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_16(tmem_S, make_smem_desc_sw128(qa + k * 32, 16, 1024), make_smem_desc_sw128(ka + k * 32, 16, 1024), idesc_s,
                  (uint32_t)(k != 0));
        umma_commit(&s_full[t]);
        if (j == nblk - 1) umma_commit(&q_empty[qb]);            // this tile's Q fully consumed
        if (++s_stage == kKvStages) { s_stage = 0; s_phase ^= 1; }
      }
    }
  } else if ((warp == 4 || warp == 5) && lane == 0) {
    // ================================ PV issuer of tile t ==========================
    const int t = warp - 4;
    const uint32_t idesc_o = make_idesc_16(BQ, HD, fp16, 0, 1);   // P (TMEM) x V (MN-major, smem)
    const int my_items = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const long long total_steps = (long long)my_items * nblk;
    const uint32_t tmem_P = tmem_base + t * TM_TILE + TM_P, tmem_O = tmem_base + t * TM_TILE + TM_O;
    int o_j = 0, o_stage = 0;
    uint32_t o_phase = 0;
    for (long long g = 0; g < total_steps; ++g) {
      const uint32_t va = smem_u32(smem + OFF_KV + o_stage * 2 * KV_BYTES + KV_BYTES);
      mbar_wait_relaxed(&kv_full[o_stage], o_phase);             // (complete long ago: this thread's own acquire of V)
      mbar_wait_quiet(&p_full[t], (uint32_t)(g & 1));             // P_t(g) in TMEM, O_t rescaled if needed
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < BKV / 16; ++k)                         // 16 keys = 8 packed TMEM columns per instruction
        umma_16_ts(tmem_O, tmem_P + k * 8, make_smem_desc_sw128(va + k * 2048, 8192, 1024), idesc_o,
                   (uint32_t)((o_j | k) != 0));
      umma_commit(&pv_done[t]);
      umma_commit(&kv_empty[o_stage]);                           // this tile is done with K_j and V_j
      if (++o_j == nblk) o_j = 0;
      if (++o_stage == kKvStages) { o_stage = 0; o_phase ^= 1; }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kSoftmaxRegs));
    // ================================ softmax warpgroups ==========================
    // One warpgroup per tile; a thread is one query row (TMEM lane) and owns its 128 keys of every step.
    const int t = (warp - kRoleWarps) / 4;         // tile
    const int quad = warp & 3;                     // TMEM lane quadrant of this warp
    const int row = quad * 32 + lane;              // query row inside the tile == TMEM lane
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    const uint32_t tmem_S = tmem_base + t * TM_TILE + TM_S + lane_off;
    const uint32_t tmem_P = tmem_base + t * TM_TILE + TM_P + lane_off;
    const uint32_t tmem_O = tmem_base + t * TM_TILE + TM_O + lane_off;
    uint8_t* srow = smem + OFF_STG + t * STG_BYTES + row * 128;
    const uint32_t b_s_full = smem_u32(&s_full[t]), b_s_free = smem_u32(&s_free[t]), b_p_full = smem_u32(&p_full[t]),
                   b_pv_done = smem_u32(&pv_done[t]);
    const float neg_masked = -10000.f;             // masked_fill value, modules.py:911-915
    long long g = 0;
    // The read-out of an item's O (its "epilogue") is deferred into the first step of the NEXT item, after that step's
    // exponentials: PV(last) of the finished item completes behind them instead of being waited for (ncu: 13 probes
    // per item on that wait = 6 % of the softmax warps' time at R = 1024, more for shallower MSAs).
    bool have_prev = false, s_ok = false;
    Item prev_it{0, 0, 0};
    float prev_l = 0.f;
    auto read_out = [&](const Item& pit, float l) {
      // 16-bit rows staged in shared memory (SWIZZLE_128B pattern of the store's tensor map), one asynchronous TMA
      // store per 32 rows.
      if (lane == 0) bulk_wait_read0();            // the staged rows of the item before have been read by their store
      __syncwarp();
      const float inv = 1.f / l;
#pragma unroll 1
      for (int hlf = 0; hlf < 2; ++hlf) {
        uint32_t ov[32];
        tmem_ld_32x32(tmem_O + hlf * 32, ov);
        tmem_ld_wait();
#pragma unroll
        for (int d = 0; d < 32; d += 8) {
          uint4 val;
          if (fp16)
            val = make_uint4(pack_f16(__uint_as_float(ov[d]) * inv, __uint_as_float(ov[d + 1]) * inv),
                             pack_f16(__uint_as_float(ov[d + 2]) * inv, __uint_as_float(ov[d + 3]) * inv),
                             pack_f16(__uint_as_float(ov[d + 4]) * inv, __uint_as_float(ov[d + 5]) * inv),
                             pack_f16(__uint_as_float(ov[d + 6]) * inv, __uint_as_float(ov[d + 7]) * inv));
          else
            val = make_uint4(pack_bf16(__uint_as_float(ov[d]) * inv, __uint_as_float(ov[d + 1]) * inv),
                             pack_bf16(__uint_as_float(ov[d + 2]) * inv, __uint_as_float(ov[d + 3]) * inv),
                             pack_bf16(__uint_as_float(ov[d + 4]) * inv, __uint_as_float(ov[d + 5]) * inv),
                             pack_bf16(__uint_as_float(ov[d + 6]) * inv, __uint_as_float(ov[d + 7]) * inv));
          const int ch = hlf * 4 + (d >> 3);
          *reinterpret_cast<uint4*>(srow + ((ch ^ (row & 7)) << 4)) = val;
        }
      }
      fence_proxy_async_smem();     // staged rows -> visible to the TMA (async proxy)
      __syncwarp();
      const int i_warp = pit.i0 + t * BQ + quad * 32;          // first query row of this warp; rows >= R are clipped
      if (lane == 0 && i_warp < R) {
        tma_store_3d(&tm_o, smem + OFF_STG + t * STG_BYTES + quad * 32 * 128, pit.h * HD, pit.c, i_warp);
        bulk_commit();
      }
    };
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const Item it = decode_item(item, nqb, H);
      float m_ref = -INFINITY, l_run = 0.f;
      for (int j = 0; j < nblk; ++j, ++g) {
        const int j0 = j * BKV;
        if (!s_ok) mbar_wait_quiet_u32(b_s_full, (uint32_t)(g & 1));   // (probed inside the previous step)
        tc_fence_after();
        uint32_t sv[BKV / 32][32];
#pragma unroll
        for (int q = 0; q < BKV / 32; ++q) tmem_ld_32x32(tmem_S + q * 32, sv[q]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(b_s_free);   // S columns may be overwritten by the next step's S

        if (pad != nullptr || j * BKV + BKV > R) {               // warp-uniform slow path: key masks
          const int n_valid = R - j0;
#pragma unroll
          for (int q = 0; q < BKV / 32; ++q) {
            uint32_t mbits = 0;
            if (pad != nullptr) {
              const int jk = j0 + q * 32 + lane;
              mbits = __ballot_sync(0xffffffffu, jk < R && pad[(size_t)jk * C + it.c] != 0);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float v = __uint_as_float(sv[q][e]);
              if ((mbits >> e) & 1u) v = neg_masked;
              if (q * 32 + e >= n_valid) v = -INFINITY;       // key row does not exist
              sv[q][e] = __float_as_uint(v);
            }
          }
        }
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int q = 0; q < BKV / 32; ++q) {
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            mx0 = fmaxf(mx0, __uint_as_float(sv[q][e]));
            mx1 = fmaxf(mx1, __uint_as_float(sv[q][e + 1]));
            mx2 = fmaxf(mx2, __uint_as_float(sv[q][e + 2]));
            mx3 = fmaxf(mx3, __uint_as_float(sv[q][e + 3]));
          }
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * kLog2e;   // log2 domain; finite (>= 1 real key)
        // lazy rescale: keep the old reference unless the max grew by more than the threshold
        float factor = 1.f;
        const bool grow = mx > m_ref + kRescaleThreshold;   // true on the first block (m_ref = -inf)
        if (grow) {
          factor = ex2(m_ref - mx);                          // 0 on the first block
          m_ref = mx;
          l_run *= factor;
        }
        const bool rescale = (j > 0) && __any_sync(0xffffffffu, grow);
        bool pv_ok = g == 0;
        // exponentials on packed fp32 pairs; the 16-bit P words (keys 2w, 2w+1 -> word w) overwrite sv[0] (and sv[1])
        // behind the read position
        const uint64_t c_l2e = f32x2_pack(kLog2e, kLog2e), c_negm = f32x2_pack(-m_ref, -m_ref);
        uint64_t acc0 = f32x2_pack(0.f, 0.f), acc1 = acc0;
#pragma unroll
        for (int q = 0; q < BKV / 32; ++q) {
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            const uint64_t x0 = f32x2_fma(f32x2_pack(__uint_as_float(sv[q][e]), __uint_as_float(sv[q][e + 1])), c_l2e, c_negm);
            const uint64_t x1 = f32x2_fma(f32x2_pack(__uint_as_float(sv[q][e + 2]), __uint_as_float(sv[q][e + 3])), c_l2e, c_negm);
            float a0, a1, a2, a3;
            f32x2_unpack(x0, a0, a1);
            a0 = ex2(a0); a1 = ex2(a1);
            if (q == BKV / 32 - 1 && e == 16) {
              // probe "PV(g-1) done" seven eighths through (a test_wait is non-blocking; its ~100 cycles of latency pass
              // behind the last exponentials; the in-kernel timeline puts PV(g-1)'s completion ~1300 cycles after P(g-1)
              // was handed over: a barrier hand-over between threads costs ~350 cycles each way)
              anchor_after(a1);
              if (g > 0) pv_ok = mbar_test_wait_u32(b_pv_done, (uint32_t)((g - 1) & 1));
            }
            f32x2_unpack(x1, a2, a3);
            a2 = ex2(a2); a3 = ex2(a3);
            acc0 = f32x2_add(acc0, f32x2_pack(a0, a1));
            acc1 = f32x2_add(acc1, f32x2_pack(a2, a3));
            const int w = (q * 32 + e) >> 1;                 // P word index inside this thread's columns
            sv[w >> 5][w & 31] = kFp16 ? pack_f16(a0, a1) : pack_bf16(a0, a1);
            sv[(w + 1) >> 5][(w + 1) & 31] = kFp16 ? pack_f16(a2, a3) : pack_bf16(a2, a3);
          }
        }
        {
          float s0, s1, s2, s3;
          f32x2_unpack(acc0, s0, s1);
          f32x2_unpack(acc1, s2, s3);
          l_run += (s0 + s1) + (s2 + s3);
        }
        s_ok = mbar_test_wait_u32(b_s_full, (uint32_t)((g + 1) & 1));   // next step's S; the answer is used ~400 cycles on
        if (!pv_ok) mbar_wait_quiet_u32(b_pv_done, (uint32_t)((g - 1) & 1));   // PV(g-1) done: P columns free, O_t stable
        tc_fence_after();
        if (j == 0 && have_prev) read_out(prev_it, prev_l);     // the finished item's O, before PV(g) overwrites it
        if (rescale) {                              // warp-uniform; rare once the max has settled
          uint32_t ov[32];
#pragma unroll 1
          for (int hlf = 0; hlf < 2; ++hlf) {
            tmem_ld_32x32(tmem_O + hlf * 32, ov);
            tmem_ld_wait();
#pragma unroll
            for (int d = 0; d < 32; ++d) ov[d] = __float_as_uint(__uint_as_float(ov[d]) * factor);
            tmem_st_32x32(tmem_O + hlf * 32, ov);
          }
        }
#pragma unroll
        for (int q = 0; q < BKV / 64; ++q) tmem_st_32x32(tmem_P + q * 32, sv[q]);   // P(g): two keys per column, A operand of P V
        tmem_st_wait();
        tc_fence_before();                          // our tcgen05.ld / st precede the MMA that follows the barrier
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(b_p_full);
      }
      prev_it = it;
      prev_l = l_run;
      have_prev = true;
    }
    if (have_prev) {                                // the last item of this CTA
      mbar_wait_quiet_u32(b_pv_done, (uint32_t)((g - 1) & 1));
      tc_fence_after();
      read_out(prev_it, prev_l);
    }
    tc_fence_before();
  }

  if (warp >= kRoleWarps && lane == 0) bulk_wait_all0();   // the last items' TMA stores have left shared memory
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

template <bool kFp16>
int launch_fa(const CUtensorMap& tq, const CUtensorMap& tkv, const CUtensorMap& to, int R, int C, int H, int col_major,
              const uint8_t* pad, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(col_attn_fa_kernel<kFp16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    attr_set = true;
  }
  const long long n_items = (long long)C * H * ((R + NT * BQ - 1) / (NT * BQ));
  RNAMSM_REQUIRE(n_items < (1LL << 31), "col_attn_fa: too many work items");
  int sms = 0, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (sms <= 0) sms = 148;
  const int grid = (int)std::min<long long>(n_items, sms);
  ProfScope prof(KC_COL_ATTN, st);
  RNAMSM_CHECK_CUDA(launch_pdl(col_attn_fa_kernel<kFp16>, dim3(grid), dim3(kThreads), kSmem, st, tq, tkv, to, R, C, H,
                               col_major, (int)n_items, pad));
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int launch_col_attn_fa_16(const void* qkv, int R, int C, int H, int fp16, int col_major, const uint8_t* pad, void* ctx,
                          cudaStream_t st) {
  RNAMSM_REQUIRE(R >= 1 && C >= 1 && H >= 1, "col_attn_fa: bad shape");
  const int ld = 3 * H * HD;
  CUtensorMap tq, tkv, to;
  // token-major q|k|v [R, C, 3D] or column-major [C, R, 3D] (rows of one column 3D elements apart: the layout the
  // forward uses, api.cu)
  uint64_t dims[3] = {(uint64_t)ld, (uint64_t)(col_major ? R : C), (uint64_t)(col_major ? C : R)};
  uint64_t strides[2] = {(uint64_t)ld * 2, (uint64_t)(col_major ? R : C) * ld * 2};
  uint32_t box_q[3] = {HD, (uint32_t)(col_major ? BQ : 1), (uint32_t)(col_major ? 1 : BQ)};
  uint32_t box_kv[3] = {HD, (uint32_t)(col_major ? BKV : 1), (uint32_t)(col_major ? 1 : BKV)};
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  if (encode_tmap(&tq, in_dt, qkv, 3, dims, strides, box_q)) return 3;
  if (encode_tmap(&tkv, in_dt, qkv, 3, dims, strides, box_kv)) return 3;
  // ctx [R, C, D] token-major: one 32-row x 64-column box per softmax warp and item
  uint64_t odims[3] = {(uint64_t)H * HD, (uint64_t)C, (uint64_t)R};
  uint64_t ostrides[2] = {(uint64_t)H * HD * 2, (uint64_t)C * H * HD * 2};
  uint32_t box_o[3] = {HD, 1, 32};
  if (encode_tmap(&to, in_dt, ctx, 3, odims, ostrides, box_o)) return 3;
  return fp16 ? launch_fa<true>(tq, tkv, to, R, C, H, col_major, pad, st)
              : launch_fa<false>(tq, tkv, to, R, C, H, col_major, pad, st);
}

}  // namespace rnamsm
