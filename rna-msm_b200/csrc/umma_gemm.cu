// 16-bit tensor-core path: one persistent, warp-specialised tcgen05 GEMM serving the three dense
// contractions of the forward, run by CTA PAIRS (cta_group::2): the two CTAs of a cluster sit on
// the two SMs of one TPC and share one 256 x 256 accumulator tile -- each CTA stages its own
// 128 rows of A and its own 128-row half of B, so per-SM operand traffic from L2 (the bound of a
// single-CTA 128 x 256 kernel: 48 KiB per k-block) drops to 32 KiB and each MMA reads both halves
// of B across the pair.  Operands come in through TMA (SWIZZLE_128B) into a 6-stage ring, are
// multiplied by tcgen05.mma.cta_group::2 (M=256, N=256, K=16 per instruction, fp32 accumulators
// in TMEM, double-buffered so the epilogue of tile t overlaps the MMAs of tile t+1) and leave
// through tcgen05.ld -> registers -> swizzled smem staging -> TMA store (coalesced, clipped at
// the tensor edge by the hardware).  The residual epilogue is a TMA reduce-add on the fp32
// stream, so the epilogue never reads global memory.
//
//   DENSE : out[m,n] = epi( sum_k x[m,k] W[n,k] + b[n] )                 nn.Linear sites,
//           modules.py:760-766 (q/k/v), :799 (out_proj), :424-426 (fc1/GELU/fc2), :314 (lm dense)
//   TIED  : partial[s,h,i,j] = sum_{r in split s} sum_d q[r,i,h,d] k[r,j,h,d]   modules.py:774
//           (K-loop walks MSA rows; one 64-wide head slice per k-block, split-K over row ranges)
//   AV    : ctx[r,i,h,:] = sum_j P[h,i,j] v[r,j,h,:]                            modules.py:797
//           (P tile is the stationary A operand; B = V read in place as an MN-major operand,
//            four MSA rows x 64 head dims per 256-wide N tile, two rows per CTA of the pair)
//
// Operand element type is bf16 or fp16 (same tensor-core rate, kind::f16); fp16 carries three more
// mantissa bits and is what the tied row-attention block uses (see api.cu).
//
//   DENSE, kTf32 : the fp32 path's nn.Linear on the tensor cores.  fp32 operands are split on the device into
//           hi = the value rounded to nearest at tf32 precision and lo = the (exact) remainder x - hi rounded likewise
//           (|x - hi - lo| <= 2^-23 |x|), and every k-step issues three tcgen05.mma kind::tf32 into the same fp32
//           accumulator: lo*hi + hi*lo + hi*hi (the dropped lo*lo term is 2^-22 of the product, of either sign) --
//           fp32-grade results at a third of the tf32 rate: measured 300 TF/s against the FFMA kernel's 37.
//
// Warp roles (384 threads per CTA): warp 0 = TMA producer (one elected lane, both CTAs), warp 1 =
// MMA issuer (one elected lane, leader CTA only), warp 2 = TMEM allocation, warp 3 idle,
// warps 4..11 = epilogue (TMEM lane quadrant = warp % 4, column half = (warp - 4) / 4).
// Pipelines: smem full/empty ring (full barriers live in the leader CTA and collect both CTAs'
// TMA bytes; empty barriers are armed in both CTAs by a multicast tcgen05.commit), TMEM
// full (multicast commit) / empty (leader barrier, remote arrivals from the peer's epilogue).
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include <stdlib.h>

#include "launch.h"

namespace rnamsm {

namespace {

constexpr int BLOCK_M = 128;                     // rows per CTA (256 per pair)
constexpr int PAIR_M = 2 * BLOCK_M;
constexpr int BLOCK_N = 256;                     // accumulator columns per pair (128 B rows staged per CTA)
constexpr int HALF_N = BLOCK_N / 2;
constexpr int BLOCK_K = 64;                      // one SWIZZLE_128B atom of 16-bit elements along K
constexpr int UMMA_K = 16;
constexpr int kStagesDefault = 6;
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KiB
constexpr int B_BYTES = HALF_N * BLOCK_K * 2;    // 16 KiB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;   // 32 KiB per CTA per k-block
constexpr int kTmemCols = 512;                   // 2 accumulator stages x 256 fp32 columns
constexpr int kEpiWarps = 8;
constexpr int kFirstEpiWarp = 4;
constexpr int kThreads = 32 * (kFirstEpiWarp + kEpiWarps);
constexpr int kLnWarps = 4;                      // LayerNorm warps of the fused residual + LayerNorm variant
constexpr int kFirstLnWarp = kFirstEpiWarp + kEpiWarps;
constexpr int kThreadsLn = kThreads + 32 * kLnWarps;
constexpr int kLnMaxVec = 8;                     // N <= 8 * 128 features per row
constexpr int kLnSlots = 4;                      // tiles the epilogue may run ahead of the LayerNorm warps
constexpr int EPI_BUF_BYTES = 32 * 128;          // one 32-row x 128 B staging box per epilogue warp
constexpr int kSmemBytes = kStagesDefault * STAGE_BYTES + kEpiWarps * EPI_BUF_BYTES + 256 + 1024;
// kWide (the fc1 + GELU instance): 16 epilogue warps, each owning 32 rows x 64 columns of the accumulator instead of
// 32 x 128, and a 5-stage operand ring so that their 16 staging boxes fit.  The GELU epilogue is ~2200 instructions per
// warp and tile with little parallelism inside a warp (ncu: issue slots 49 % busy at two epilogue warps per scheduler);
// at 8 warps it takes about as long as the 12 k-blocks of the tile's MMAs and the tensor pipe waits for its accumulator
// buffer (fc1 1181 TF/s vs 1332 with the bias-only epilogue, tools/epi_cost_bench.py).
constexpr int kEpiWarpsWide = 16;
constexpr int kThreadsWide = 32 * (kFirstEpiWarp + kEpiWarpsWide);
constexpr int kStagesWide = 5;
static_assert(kStagesWide * STAGE_BYTES + kEpiWarpsWide * EPI_BUF_BYTES == kStagesDefault * STAGE_BYTES + kEpiWarps * EPI_BUF_BYTES,
              "the wide-epilogue variant uses the same shared-memory footprint");

enum { V_DENSE = 0, V_TIED = 1, V_AV = 2 };

struct GemmArgs {
  int m_tiles, n_tiles, batches, splits;
  int k_blocks;          // DENSE: K/64, AV: ceil(C/64); TIED: rows of the split (computed per tile)
  int M, N;              // logical bounds for the epilogue (DENSE: M x N; TIED: C x C; AV: C x R)
  int R, C, H;
  int rows_per_split;
  int epi_kind;
  int fp16;              // operand / 16-bit output element type: 0 = bf16, 1 = fp16
  const float* bias;
  float q_scale;
  int q_cols;
  const uint8_t* row_mask;
  void* out;             // TIED only (direct fp32 stores); the other variants store through tmap_out
  int ld_out;
  // residual epilogue into PEER memory (sharded forward, column block's out-projection): output row
  // m = r * Cn + c_local of this rank's column shard is reduce-added into row (r % Rn) * C + c0 + c_local
  // of the fp32 residual stream of rank r / Rn, through that rank's tensor map.
  int peer_n, peer_Rn, peer_Cn, peer_c0, peer_box_rows;
  int m_tile_shift;      // DENSE: m-tile order rotated by this (per-rank) so ranks scatter to different owners at once
  // fused residual + LayerNorm (kLN variant): y = LN(out) over full rows of N features, written in 16 bits
  const float* ln_w;
  const float* ln_b;
  void* ln_out;
  float ln_eps;
  int ln_fp16;           // element type of ln_out: 0 = bf16, 1 = fp16
  int ln_tr_R, ln_tr_C;  // > 0: output row (m % tr_C) * tr_R + m / tr_C (column-major token order)
  int* ln_counters;      // [2 * m_tiles] zero on entry, zero again on exit: arrivals per (m-block, CTA rank)
  int ln_debug;          // RNAMSM_LN_DEBUG bits (experiments): 1 skip the row work, 2 read rows half a tensor away,
                         // 4 plain (L1-cached) loads, 8 no stores
};

struct PeerMaps { CUtensorMap m[RNAMSM_MAX_PEERS]; };

struct TileCoord {
  int m0, n0;            // element offsets of the PAIR tile inside the logical M / N extents
  int batch, split;
  int kb_begin, kb_count;
};

template <int kVariant, int kBN>
__device__ __forceinline__ TileCoord decode_tile(const GemmArgs& g, int tile) {
  TileCoord t;
  if (kVariant == V_DENSE) {
    t.n0 = (tile % g.n_tiles) * kBN;
    int mt = tile / g.n_tiles + g.m_tile_shift;
    if (mt >= g.m_tiles) mt -= g.m_tiles;
    t.m0 = mt * PAIR_M;
    t.batch = 0; t.split = 0; t.kb_begin = 0; t.kb_count = g.k_blocks;
  } else if (kVariant == V_TIED) {
    t.n0 = (tile % g.n_tiles) * kBN;  tile /= g.n_tiles;
    t.m0 = (tile % g.m_tiles) * PAIR_M;   tile /= g.m_tiles;
    t.split = tile % g.splits;
    t.batch = tile / g.splits;
    t.kb_begin = t.split * g.rows_per_split;
    t.kb_count = min(g.R, t.kb_begin + g.rows_per_split) - t.kb_begin;
  } else {
    t.m0 = (tile % g.m_tiles) * PAIR_M;   tile /= g.m_tiles;
    t.n0 = (tile % g.n_tiles) * 4;        // first MSA row of the 4-row group
    t.batch = tile / g.n_tiles;
    t.split = 0; t.kb_begin = 0; t.kb_count = g.k_blocks;
  }
  return t;
}

// Persistent tile order: tile = pair + lt * n_pairs, so the n-tiles of one m-block run on neighbouring pairs at the same
// time and share the block's A rows through L2 (giving a pair whole m-blocks instead re-reads A from HBM once its 74
// concurrent copies outgrow L2: measured 1219 -> 944 TF/s on fc2).
__device__ __forceinline__ int tile_at(int lt, int pair, int n_pairs, int total_tiles) {
  const long long t = (long long)pair + (long long)lt * n_pairs;
  return t < total_tiles ? (int)t : -1;
}

// erf-GELU for the 16-bit epilogue: erfc(z) ~= (1 + a1 z + ... + a6 z^6)^-16 (Abramowitz & Stegun
// 7.1.28, |error| <= 3e-7 -- far below the 16-bit output rounding), one MUFU.RCP + ~14 FMA-class
// instructions per element instead of erff's ~30, which keeps the fc1 epilogue under the MMA time
// of its tile.  The fp32 parity path keeps erff (simt_f32.cu).
__device__ __forceinline__ float gelu_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  float p = fmaf(z, 0.0000430638f, 0.0002765672f);
  p = fmaf(p, z, 0.0001520143f);
  p = fmaf(p, z, 0.0092705272f);
  p = fmaf(p, z, 0.0422820123f);
  p = fmaf(p, z, 0.0705230784f);
  p = fmaf(p, z, 1.0f);
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
  r *= r; r *= r; r *= r; r *= r;       // erfc(z)
  const float h = 0.5f * x * r;
  return x >= 0.f ? x - h : h;
}

// Two erf-GELUs at once on packed fp32 pairs (FFMA2 / FMUL2 / FADD2): gelu(x) = 0.5 (x + |x| (1 - erfc(|x|/sqrt2))),
// same A&S 7.1.28 erfc as gelu_fast.  ~19 issue slots per pair instead of ~36: the fc1 epilogue is issue-bound.
__device__ __forceinline__ void gelu_fast2(float& x0, float& x1) {
  const uint64_t x = f32x2_pack(x0, x1);
  const uint64_t ax = x & 0x7fffffff7fffffffull;                              // |x|
  const uint64_t z = f32x2_mul(ax, f32x2_pack(0.70710678118654752440f, 0.70710678118654752440f));
  uint64_t p = f32x2_fma(z, f32x2_pack(0.0000430638f, 0.0000430638f), f32x2_pack(0.0002765672f, 0.0002765672f));
  p = f32x2_fma(p, z, f32x2_pack(0.0001520143f, 0.0001520143f));
  p = f32x2_fma(p, z, f32x2_pack(0.0092705272f, 0.0092705272f));
  p = f32x2_fma(p, z, f32x2_pack(0.0422820123f, 0.0422820123f));
  p = f32x2_fma(p, z, f32x2_pack(0.0705230784f, 0.0705230784f));
  p = f32x2_fma(p, z, f32x2_pack(1.0f, 1.0f));
  float p0, p1, r0, r1;
  f32x2_unpack(p, p0, p1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
  uint64_t r = f32x2_pack(r0, r1);
  r = f32x2_mul(r, r); r = f32x2_mul(r, r); r = f32x2_mul(r, r); r = f32x2_mul(r, r);   // erfc(z)
  const uint64_t t = f32x2_fma(r, f32x2_pack(-1.0f, -1.0f), f32x2_pack(1.0f, 1.0f));  // 1 - erfc
  const uint64_t u = f32x2_fma(ax, t, x);                                              // x + |x| (1 - erfc)
  f32x2_unpack(f32x2_mul(u, f32x2_pack(0.5f, 0.5f)), x0, x1);
}

__device__ __forceinline__ uint32_t pack16(float lo, float hi, int fp16) {
  uint32_t r;
  if (fp16)
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else
    asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// One 32-row x 128-byte box: lane `lane` writes its own row (8 x 16 B) into the SWIZZLE_128B
// staging layout (16-byte chunk c of row r lives at chunk c ^ (r & 7)): conflict-free.
__device__ __forceinline__ void stage_row(uint8_t* buf, int lane, const uint32_t (&w)[32]) {
  uint8_t* row = buf + lane * 128;
#pragma unroll
  for (int c = 0; c < 8; ++c)
    *reinterpret_cast<uint4*>(row + ((c ^ (lane & 7)) << 4)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}

// kBN = accumulator columns of the pair tile (256; 128 / 64 for the tied logits of short alignments, where a
// 256-wide tile would be mostly padding): each CTA stages kBN / 2 rows of B, TMEM holds 2 x kBN columns.
template <int kVariant, int kBN, bool kLN = false, bool kTf32 = false, bool kWide = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kLN ? kThreadsLn : (kWide ? kThreadsWide : kThreads), 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out, const GemmArgs g,
                 const __grid_constant__ PeerMaps peers) {
  constexpr int BN = kBN, HN = kBN / 2;
  // bytes per CTA per k-block: A + B tiles (16-bit: 64 elements of K per 128 B row); kTf32: hi and lo tiles of both
  // operands (fp32: 32 elements of K per 128 B row) in a shallower ring
  constexpr int STG = kTf32 ? 4 * A_BYTES : A_BYTES + HN * BLOCK_K * 2;
  constexpr int kStages = kTf32 ? 3 : (kWide ? kStagesWide : kStagesDefault);
  constexpr int EPW = kWide ? kEpiWarpsWide : kEpiWarps;   // epilogue warps per CTA
  constexpr int CW = kBN / (EPW / 4);                      // accumulator columns per epilogue warp (128; wide: 64)
  static_assert(!kWide || ((kVariant == V_DENSE || kVariant == V_AV) && kBN == BLOCK_N && !kLN && !kTf32),
                "wide epilogue: the 16-bit-output variants only");
  constexpr int KB_ELEMS = kTf32 ? 32 : BLOCK_K;         // K elements per k-block
  static_assert(!kTf32 || (kVariant == V_DENSE && kBN == BLOCK_N && !kLN), "tf32 split: the dense 256-wide variant only");
  constexpr int TMC = 2 * kBN;                           // TMEM columns (power of two >= 32)
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024 B alignment (descriptor base_offset = 0).  The dynamic smem
  // window starts at the same offset in both CTAs, so the carve-up below is identical in the pair.
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* epi_smem = smem + kStages * STG;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_smem + EPW * EPI_BUF_BYTES);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* ln_ready = tmem_empty + 2;             // [kLnSlots] kLN: this CTA's reduce-adds of a tile have been performed
  uint64_t* ln_free = ln_ready + kLnSlots;         // [kLnSlots] kLN: the LayerNorm warps are done with that slot
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(ln_free + kLnSlots);
  volatile int* ln_job = reinterpret_cast<volatile int*>(tmem_ptr + 1);   // [2] kLN: "this tile completed its m-block"

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int total_tiles = g.m_tiles * g.n_tiles * g.batches * g.splits;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if (kVariant != V_TIED) tma_prefetch_desc(&tmap_out);
  }
  if (warp == 1 && elect_one()) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 2);                 // one arrive.expect_tx per CTA of the pair (leader's copy is used)
      mbar_init(&empty_bar[s], 1);                // multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);                // multicast tcgen05.commit
      mbar_init(&tmem_empty[a], 2 * EPW);         // epilogue warps of both CTAs (leader's copy is used)
    }
    for (int a = 0; a < kLnSlots; ++a) {
      mbar_init(&ln_ready[a], kEpiWarps);         // this CTA's epilogue warps
      mbar_init(&ln_free[a], kLnWarps);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc2(tmem_ptr, TMC);
    tmem_relinquish2();
  }
  tc_fence_before();
  __syncthreads();   // CTA-local ordering of the tcgen05.alloc result (also what compute-sanitizer racecheck models)
  cluster_sync();    // both CTAs' barriers initialised and TMEM allocated before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_launch_dependents();   // this CTA holds its shared memory and TMEM: the next kernel may begin its own prologue
  pdl_wait();                // everything above overlapped the predecessor's tail; its results are needed from here on

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int lt = 0, tile; (tile = tile_at(lt, pair, n_pairs, total_tiles)) >= 0; ++lt) {
        const TileCoord t = decode_tile<kVariant, kBN>(g, tile);
        for (int kb = 0; kb < t.kb_count; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * STG;
          uint8_t* sb = sa + A_BYTES;
          const uint32_t bar = mapa_u32(smem_u32(&full_bar[stage]), 0);   // the leader's full barrier
          mbar_expect_tx_cluster(bar, STG);
          if (kTf32) {            // [A hi | A lo | B hi | B lo], the lo operands through peers.m[0] / m[1]
            tma_load_3d_2sm(sa, &tmap_a, bar, kb * KB_ELEMS, t.m0 + cta_rank * BLOCK_M, 0);
            tma_load_3d_2sm(sa + A_BYTES, &peers.m[0], bar, kb * KB_ELEMS, t.m0 + cta_rank * BLOCK_M, 0);
            tma_load_3d_2sm(sa + 2 * A_BYTES, &tmap_b, bar, kb * KB_ELEMS, t.n0 + cta_rank * HN, 0);
            tma_load_3d_2sm(sa + 3 * A_BYTES, &peers.m[1], bar, kb * KB_ELEMS, t.n0 + cta_rank * HN, 0);
          } else if (kVariant == V_DENSE) {
            tma_load_3d_2sm(sa, &tmap_a, bar, kb * BLOCK_K, t.m0 + cta_rank * BLOCK_M, 0);
            tma_load_3d_2sm(sb, &tmap_b, bar, kb * BLOCK_K, t.n0 + cta_rank * HN, 0);
          } else if (kVariant == V_TIED) {
            const int r = t.kb_begin + kb;
            tma_load_3d_2sm(sa, &tmap_a, bar, t.batch * 64, t.m0 + cta_rank * BLOCK_M, r);
            tma_load_3d_2sm(sb, &tmap_b, bar, (g.H + t.batch) * 64, t.n0 + cta_rank * HN, r);
          } else {
            tma_load_3d_2sm(sa, &tmap_a, bar, kb * BLOCK_K, t.m0 + cta_rank * BLOCK_M, t.batch);
            tma_load_3d_2sm(sb, &tmap_b, bar, (2 * g.H + t.batch) * 64, kb * BLOCK_K, t.n0 + cta_rank * 2);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA) =====================
    if (leader && elect_one()) {
      const uint32_t idesc = kTf32 ? make_idesc_tf32(PAIR_M, BN) : make_idesc_16(PAIR_M, BN, g.fp16, 0, kVariant == V_AV ? 1 : 0);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int lt = 0, tile; (tile = tile_at(lt, pair, n_pairs, total_tiles)) >= 0; ++lt) {
        const TileCoord t = decode_tile<kVariant, kBN>(g, tile);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < t.kb_count; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * STG);
          const uint32_t b_addr = a_addr + A_BYTES;
          if (kTf32) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {            // 32 fp32 per row = 4 k-steps of 8 (32 B each)
              const uint64_t a_hi = make_smem_desc_sw128(a_addr + k * 32, 16, 1024);
              const uint64_t a_lo = make_smem_desc_sw128(a_addr + A_BYTES + k * 32, 16, 1024);
              const uint64_t b_hi = make_smem_desc_sw128(a_addr + 2 * A_BYTES + k * 32, 16, 1024);
              const uint64_t b_lo = make_smem_desc_sw128(a_addr + 3 * A_BYTES + k * 32, 16, 1024);
              umma_tf32_2sm(d_tmem, a_lo, b_hi, idesc, (uint32_t)((kb | k) != 0));   // small terms first
              umma_tf32_2sm(d_tmem, a_hi, b_lo, idesc, 1u);
              umma_tf32_2sm(d_tmem, a_hi, b_hi, idesc, 1u);
            }
          } else
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // A: K-major, 128 B rows, 8-row groups 1024 B apart; +32 B per 16-element k step.
            const uint64_t adesc = make_smem_desc_sw128(a_addr + k * (UMMA_K * 2), 16, 1024);
            uint64_t bdesc;
            if (kVariant == V_AV)  // B: MN-major [2 r][64 j][64 d]: 64-wide N chunks 8 KiB apart,
              bdesc = make_smem_desc_sw128(b_addr + k * (UMMA_K * 128), 64 * 128, 1024);  // 8-row k groups 1 KiB
            else
              bdesc = make_smem_desc_sw128(b_addr + k * (UMMA_K * 2), 16, 1024);
            umma_16_2sm(d_tmem, adesc, bdesc, idesc, (uint32_t)((kb | k) != 0));
          }
          umma_commit_2sm(&empty_bar[stage]);  // both CTAs' smem slots reusable once these MMAs have read them
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[acc]);      // accumulator complete -> epilogue warps of both CTAs
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= kFirstEpiWarp && warp < kFirstEpiWarp + EPW) {
    // ================================ epilogue (both CTAs) ========================
    const int quad = warp & 3;                       // TMEM lanes [32*quad, 32*quad+32)
    const int half = (warp - kFirstEpiWarp) >> 2;    // accumulator columns [CW*half, CW*half+CW)
    uint8_t* buf = epi_smem + (warp - kFirstEpiWarp) * EPI_BUF_BYTES;
    const uint32_t empty_remote = mapa_u32(smem_u32(&tmem_empty[0]), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    int n_local = 0;
    auto ln_signal = [&](int i) {                    // lane 0: this warp's reduce-adds of local tile i are done
      const int slot = i % kLnSlots, use = i / kLnSlots;
      if (use > 0) mbar_wait(&ln_free[slot], (uint32_t)((use - 1) & 1));   // slot consumed kLnSlots tiles ago
      mbar_arrive(&ln_ready[slot]);
    };
    for (int lt = 0, tile; (tile = tile_at(lt, pair, n_pairs, total_tiles)) >= 0; ++lt) {
      n_local = lt + 1;
      const TileCoord t = decode_tile<kVariant, kBN>(g, tile);
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN + half * CW + ((uint32_t)(quad * 32) << 16);
      const int row0 = t.m0 + cta_rank * BLOCK_M + quad * 32;   // first logical row of this warp's box
      auto release_acc = [&]() {                     // every tcgen05.ld of this tile has completed
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(empty_remote + acc * 8);
      };

      if (kVariant == V_TIED) {
        // fp32 partial logits, direct stores (C need not be a multiple of 4)
        const int i = row0 + lane;
#pragma unroll 1
        for (int c = 0; c < CW / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
          if (c == CW / 32 - 1) release_acc();
          const int j0 = t.n0 + half * CW + c * 32;
          if (i >= g.C || j0 >= g.C) continue;
          float* dst = reinterpret_cast<float*>(g.out) + (((size_t)t.split * g.H + t.batch) * g.C + i) * g.C + j0;
          if ((g.C & 3) == 0 && j0 + 32 <= g.C) {
#pragma unroll
            for (int k = 0; k < 32; k += 4)
              *reinterpret_cast<float4*>(dst + k) = make_float4(__uint_as_float(v[k]), __uint_as_float(v[k + 1]),
                                                                __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]));
          } else {
#pragma unroll
            for (int k = 0; k < 32; ++k)
              if (j0 + k < g.C) dst[k] = __uint_as_float(v[k]);
          }
        }
      } else if (kVariant == V_DENSE && g.epi_kind == RNAMSM_EPI_BIAS_RESIDUAL) {
        // out(fp32) += acc + bias: 32-column boxes, TMA reduce-add into the residual stream
#pragma unroll 1
        for (int c = 0; c < CW / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
          if (c == CW / 32 - 1) release_acc();
          const int n = t.n0 + half * CW + c * 32;
          if (n >= g.N || row0 >= g.M) {
            if (kLN && lane == 0) bulk_commit();       // an empty group: every tile commits exactly CW / 32 groups
            continue;
          }
#pragma unroll
          for (int k = 0; k < 32; k += 4) {
            const float4 b = *reinterpret_cast<const float4*>(g.bias + n + k);
            v[k] = __float_as_uint(__uint_as_float(v[k]) + b.x);
            v[k + 1] = __float_as_uint(__uint_as_float(v[k + 1]) + b.y);
            v[k + 2] = __float_as_uint(__uint_as_float(v[k + 2]) + b.z);
            v[k + 3] = __float_as_uint(__uint_as_float(v[k + 3]) + b.w);
          }
          if (lane == 0) bulk_wait_read0();            // the previous box has left the staging buffer
          __syncwarp();
          stage_row(buf, lane, v);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (kVariant == V_DENSE && g.peer_n > 0) {
              // GEMM + column->row all-to-all + residual add in one: each sub-box of rows that share an
              // MSA row goes to the residual stream of the rank owning that row, over NVLink
              for (int sb = 0; sb < 32; sb += g.peer_box_rows) {
                const int m = row0 + sb;
                if (m >= g.M) break;
                const int r = m / g.peer_Cn, cl = m - r * g.peer_Cn;
                const int owner = r / g.peer_Rn;
                tma_reduce_add_3d(&peers.m[owner], buf + sb * 128, n, g.peer_c0 + cl, r - owner * g.peer_Rn);
              }
            } else {
              tma_reduce_add_3d(&tmap_out, buf, n, row0, 0);
            }
            bulk_commit();
          }
        }
        if (kLN && lt > 0 && lane == 0) {
          // all but this tile's CW / 32 groups are complete = the PREVIOUS tile's reduce-adds have been performed at
          // L2 (not merely read out of the staging buffer): tell the LayerNorm warps, one tile late and without stalling
          bulk_wait_pending<CW / 32>();
          ln_signal(lt - 1);
        }
      } else if (kTf32) {
        // fp32 outputs (bias, q scale / row mask, exact erf-GELU as in the FFMA path): 32-column boxes, TMA store
#pragma unroll 1
        for (int c = 0; c < CW / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
          if (c == CW / 32 - 1) release_acc();
          const int n = t.n0 + half * CW + c * 32;
          if (n >= g.N || row0 >= g.M) continue;
          float s = 1.f;
          if (g.epi_kind == RNAMSM_EPI_BIAS && n < g.q_cols) {   // q_cols is a multiple of 64
            const int m = row0 + lane;
            s = (g.row_mask && m < g.M && g.row_mask[m]) ? 0.f : g.q_scale;
          }
          const bool gelu = g.epi_kind == RNAMSM_EPI_BIAS_GELU;
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            float a = __uint_as_float(v[k]) + g.bias[n + k];
            a = gelu ? gelu_erf(a) : a * s;
            v[k] = __float_as_uint(a);
          }
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
          stage_row(buf, lane, v);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&tmap_out, buf, n, row0, 0);
            bulk_commit();
          }
        }
      } else {
        // 16-bit outputs: 64-column boxes (128 B rows), TMA store
#pragma unroll 1
        for (int c = 0; c < CW / 64; ++c) {
          uint32_t v0[32], v1[32];
          tmem_ld_32x32(taddr + c * 64, v0);
          tmem_ld_32x32(taddr + c * 64 + 32, v1);
          tmem_ld_wait();
          if (c == CW / 64 - 1) release_acc();
          uint32_t w[32];
          int c0, c1, c2;
          if (kVariant == V_DENSE) {
            const int n = t.n0 + half * CW + c * 64;
            if (n >= g.N || row0 >= g.M) continue;
            float s = 1.f;
            if (g.epi_kind == RNAMSM_EPI_BIAS && n < g.q_cols) {   // q_cols is a multiple of 64
              const int m = row0 + lane;
              s = (g.row_mask && m < g.M && g.row_mask[m]) ? 0.f : g.q_scale;
            }
            const bool gelu = g.epi_kind == RNAMSM_EPI_BIAS_GELU;
#pragma unroll
            for (int k = 0; k < 32; k += 4) {
              const float4 b0 = *reinterpret_cast<const float4*>(g.bias + n + k);
              const float4 b1 = *reinterpret_cast<const float4*>(g.bias + n + 32 + k);
              float a[8] = {__uint_as_float(v0[k]) + b0.x, __uint_as_float(v0[k + 1]) + b0.y,
                            __uint_as_float(v0[k + 2]) + b0.z, __uint_as_float(v0[k + 3]) + b0.w,
                            __uint_as_float(v1[k]) + b1.x, __uint_as_float(v1[k + 1]) + b1.y,
                            __uint_as_float(v1[k + 2]) + b1.z, __uint_as_float(v1[k + 3]) + b1.w};
              if (gelu) {
#pragma unroll
                for (int e = 0; e < 8; e += 2) gelu_fast2(a[e], a[e + 1]);
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) a[e] *= s;
              }
              w[k / 2] = pack16(a[0], a[1], g.fp16);
              w[k / 2 + 1] = pack16(a[2], a[3], g.fp16);
              w[16 + k / 2] = pack16(a[4], a[5], g.fp16);
              w[16 + k / 2 + 1] = pack16(a[6], a[7], g.fp16);
            }
            c0 = n; c1 = row0; c2 = 0;
          } else {  // V_AV: columns = (MSA row r, 64 head dims); rows = query column i
            const int r = t.n0 + half * (CW / 64) + c;
            if (r >= g.R || row0 >= g.C) continue;
#pragma unroll
            for (int k = 0; k < 32; k += 2) {
              w[k / 2] = pack16(__uint_as_float(v0[k]), __uint_as_float(v0[k + 1]), g.fp16);
              w[16 + k / 2] = pack16(__uint_as_float(v1[k]), __uint_as_float(v1[k + 1]), g.fp16);
            }
            c0 = t.batch * 64; c1 = row0; c2 = r;
          }
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
          stage_row(buf, lane, w);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (kVariant == V_DENSE && g.peer_n > 0) {
              // 16-bit result rows stored into the row owners' receive buffers over NVLink (half the bytes
              // of the fp32 reduce; the add happens in the owner's next LayerNorm pass)
              for (int sb = 0; sb < 32; sb += g.peer_box_rows) {
                const int m = c1 + sb;
                if (m >= g.M) break;
                const int r = m / g.peer_Cn, cl = m - r * g.peer_Cn;
                const int owner = r / g.peer_Rn;
                tma_store_3d(&peers.m[owner], buf + sb * 128, c0, g.peer_c0 + cl, r - owner * g.peer_Rn);
              }
            } else {
              tma_store_3d(&tmap_out, buf, c0, c1, c2);
            }
            bulk_commit();
          }
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) {
      bulk_wait_all0();                // our global writes are complete before the CTA retires
      if (kLN && n_local > 0) ln_signal(n_local - 1);
    }
  } else if (kLN && warp >= kFirstLnWarp) {
    // ================================ LayerNorm of the finished rows (both CTAs) ====
    // An m-block's N / 256 column tiles are reduce-added into the fp32 residual stream by neighbouring pairs.  Each CTA
    // counts its finished tiles per (m-block, CTA rank) in global memory; the CTA whose arrival completes the block
    // ("last arriver", the threadFenceReduction pattern) owns the LayerNorm of those 128 rows: it reads them back from
    // L2 (ld.global.cg -- they were just written there), normalises over the full N features with fp32 statistics
    // (same code as layernorm_kernel) and writes the 16-bit operand of the next GEMM.  The stand-alone LayerNorm pass
    // (3 KiB read + 1.5 KiB written per token from HBM) disappears.
    const int w = warp - kFirstLnWarp;
    const int nv = g.N >> 7;
    const float* xs = reinterpret_cast<const float*>(g.out);
    for (int lt = 0, tile; (tile = tile_at(lt, pair, n_pairs, total_tiles)) >= 0; ++lt) {
      const TileCoord t = decode_tile<kVariant, kBN>(g, tile);
      const int slot = lt % kLnSlots, use = lt / kLnSlots;
      mbar_wait(&ln_ready[slot], (uint32_t)(use & 1));
      if (w == 0 && lane == 0) {
        int* cnt = g.ln_counters + 2 * (t.m0 / PAIR_M) + (int)cta_rank;
        __threadfence();                              // our CTA's (completed) reduce-adds before the arrival
        const int last = atomicAdd(cnt, 1) == g.n_tiles - 1;
        if (last) {
          *cnt = 0;                                   // nobody else touches this counter again: clean for the next launch
          __threadfence();                            // the other CTAs' arrivals (and their rows) before our reads
        }
        ln_job[lt & 1] = last;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kLnWarps) : "memory");   // the LayerNorm warps only
      if (ln_job[lt & 1] && !(g.ln_debug & 1)) {
        fence_proxy_async_all();                      // async-proxy (TMA reduce) writes -> our generic-proxy loads
        const int row_base = t.m0 + (int)cta_rank * BLOCK_M + w * (BLOCK_M / kLnWarps);
#pragma unroll 1
        for (int rr = 0; rr < BLOCK_M / kLnWarps; rr += 2) {           // two rows in flight per warp
          const long long row = row_base + rr;
          if (row >= g.M) break;
          const bool two = row + 1 < g.M;
          const long long rsrc = (g.ln_debug & 2) ? (row + g.M / 2) % (g.M - 1) : row;
          const float* src = xs + (size_t)rsrc * g.N;
          const float* src1 = two ? src + g.N : src;      // single tail row: read it twice, never out of bounds
          float4 v0[kLnMaxVec], v1[kLnMaxVec];
          if (g.ln_debug & 4) {
#pragma unroll
            for (int i = 0; i < kLnMaxVec; ++i)
              if (i < nv) {
                v0[i] = *reinterpret_cast<const float4*>(src + lane * 4 + i * 128);
                v1[i] = *reinterpret_cast<const float4*>(src1 + lane * 4 + i * 128);
              }
          } else {
#pragma unroll
            for (int i = 0; i < kLnMaxVec; ++i)
              if (i < nv) {
                v0[i] = __ldcg(reinterpret_cast<const float4*>(src + lane * 4 + i * 128));
                v1[i] = __ldcg(reinterpret_cast<const float4*>(src1 + lane * 4 + i * 128));
              }
          }
          warp_layernorm2(v0, v1, nv, g.N, g.ln_eps, g.ln_w, g.ln_b, lane);
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            if ((q == 1 && !two) || (g.ln_debug & 8)) break;
            const long long rw = row + q;
            const long long orow = g.ln_tr_C > 0 ? (rw % g.ln_tr_C) * g.ln_tr_R + rw / g.ln_tr_C : rw;
            uint16_t* dst = reinterpret_cast<uint16_t*>(g.ln_out) + (size_t)orow * g.N;
#pragma unroll
            for (int i = 0; i < kLnMaxVec; ++i)
              if (i < nv) {
                const float4 y = q == 0 ? v0[i] : v1[i];
                *reinterpret_cast<uint2*>(dst + lane * 4 + i * 128) =
                    make_uint2(pack16(y.x, y.y, g.ln_fp16), pack16(y.z, y.w, g.ln_fp16));
              }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ln_free[slot]);
    }
  }

  tc_fence_before();
  cluster_sync();   // the peer's smem / barriers stay valid until both CTAs are done
  if (warp == 2) tmem_dealloc2(tmem_base, TMC);
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// CTA pairs that can be co-resident: a persistent grid must not exceed it (a pair that only starts
// once another has finished its whole share would double the kernel time).  Not every GPC has an
// even number of usable SMs, so this can be below num_sms() / 2.
int g_max_pairs = 0;

// Resolved ONCE per process, before anything is planned or launched, so that every workspace plan and every launch
// of the process sees the same value (the split count of the tied logits depends on it).  All variants of the kernel
// have the same block size and dynamic shared memory, hence the same cluster occupancy: the DENSE instance is queried.
static void ensure_max_pairs() {
  if (g_max_pairs != 0) return;
  cudaFuncSetAttribute(umma_gemm_kernel<V_DENSE, BLOCK_N>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(num_sms(), 1, 1);
  cfg.blockDim = dim3(kThreads, 1, 1);
  cfg.dynamicSmemBytes = kSmemBytes;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  int n = 0;
  cudaError_t e = cudaOccupancyMaxActiveClusters(&n, umma_gemm_kernel<V_DENSE, BLOCK_N>, &cfg);
  if (e != cudaSuccess || n <= 0) { cudaGetLastError(); n = num_sms() / 2; }
  const char* env = getenv("RNAMSM_GEMM_PAIRS");
  if (env && atoi(env) > 0) n = atoi(env);
  g_max_pairs = std::max(1, std::min(n, num_sms() / 2));
}

template <int kVariant, int kBN = BLOCK_N, bool kLN = false, bool kTf32 = false, bool kWide = false>
int launch_variant(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const GemmArgs& g,
                   int prof_class, cudaStream_t st, const PeerMaps* peers = nullptr) {
  static bool attr_set = false;
  if (!attr_set) {
    RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(umma_gemm_kernel<kVariant, kBN, kLN, kTf32, kWide>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           kSmemBytes));
    attr_set = true;
  }
  ensure_max_pairs();
  const long long total = (long long)g.m_tiles * g.n_tiles * g.batches * g.splits;
  RNAMSM_REQUIRE(total > 0 && total < (1LL << 31), "umma_gemm: tile count %lld out of range", total);
  const int pairs = (int)std::min<long long>(total, g_max_pairs);
  ProfScope prof(prof_class, st);
  static const PeerMaps no_peers{};
  RNAMSM_CHECK_CUDA(launch_pdl(umma_gemm_kernel<kVariant, kBN, kLN, kTf32, kWide>, dim3(2 * pairs),
                               dim3(kLN ? kThreadsLn : (kWide ? kThreadsWide : kThreads)), kSmemBytes, st, ta, tb, to, g,
                               peers ? *peers : no_peers));
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
int launch_linear_16(const void* x, const void* W, long long M, int N, int K, int fp16, const LinearEpilogue& epi,
                     void* out, cudaStream_t st, const LnFuse* ln) {
  RNAMSM_REQUIRE(M > 0 && M < (1LL << 31), "linear_16: M=%lld out of range", M);
  RNAMSM_REQUIRE(N % 64 == 0 && K % BLOCK_K == 0 && K >= BLOCK_K, "linear_16: N=%d and K=%d must be multiples of 64", N, K);
  RNAMSM_REQUIRE(epi.bias != nullptr, "linear_16: bias required");
  RNAMSM_REQUIRE(epi.q_cols % 64 == 0, "linear_16: q_cols=%d must be a multiple of 64", epi.q_cols);
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  CUtensorMap ta, tb, to;
  {
    uint64_t dims[3] = {(uint64_t)K, (uint64_t)M, 1};
    uint64_t strides[2] = {(uint64_t)K * 2, (uint64_t)M * K * 2};
    uint32_t box[3] = {BLOCK_K, BLOCK_M, 1};
    if (encode_tmap(&ta, in_dt, x, 3, dims, strides, box)) return 3;
  }
  {
    uint64_t dims[3] = {(uint64_t)K, (uint64_t)N, 1};
    uint64_t strides[2] = {(uint64_t)K * 2, (uint64_t)N * K * 2};
    uint32_t box[3] = {BLOCK_K, HALF_N, 1};
    if (encode_tmap(&tb, in_dt, W, 3, dims, strides, box)) return 3;
  }
  if (epi.kind == RNAMSM_EPI_BIAS_RESIDUAL) {
    uint64_t dims[3] = {(uint64_t)N, (uint64_t)M, 1};
    uint64_t strides[2] = {(uint64_t)N * 4, (uint64_t)M * N * 4};
    uint32_t box[3] = {32, 32, 1};
    if (encode_tmap(&to, TMAP_F32, out, 3, dims, strides, box)) return 3;
  } else {
    uint64_t dims[3] = {(uint64_t)N, (uint64_t)M, 1};
    uint64_t strides[2] = {(uint64_t)N * 2, (uint64_t)M * N * 2};
    uint32_t box[3] = {64, 32, 1};
    if (encode_tmap(&to, in_dt, out, 3, dims, strides, box)) return 3;
  }
  GemmArgs g{};
  g.m_tiles = ceil_div(M, PAIR_M);
  g.n_tiles = ceil_div(N, BLOCK_N);
  g.batches = 1; g.splits = 1;
  g.k_blocks = K / BLOCK_K;
  g.M = (int)M; g.N = N;
  g.fp16 = fp16;
  g.epi_kind = epi.kind; g.bias = epi.bias; g.q_scale = epi.q_scale; g.q_cols = epi.q_cols; g.row_mask = epi.row_mask;
  g.out = out; g.ld_out = N;
  if (ln != nullptr) {
    // fused residual + LayerNorm: the CTA whose reduce-adds complete an m-block's rows reads them back from L2 and
    // emits LayerNorm(row) as the 16-bit operand of the next GEMM (NormalizedResidualBlock, modules.py:385-401)
    RNAMSM_REQUIRE(epi.kind == RNAMSM_EPI_BIAS_RESIDUAL, "linear_16: LayerNorm fusion needs the residual epilogue");
    RNAMSM_REQUIRE(N % 128 == 0 && N <= 128 * kLnMaxVec, "linear_16: LayerNorm fusion needs N=%d to be a multiple of 128 <= 1024", N);
    RNAMSM_REQUIRE(ln->w && ln->b && ln->out && ln->out != out && ln->counters,
                   "linear_16: LayerNorm fusion needs weight, bias, a separate output and the (zeroed) arrival counters");
    RNAMSM_REQUIRE(ln->tr_C <= 0 || (long long)ln->tr_R * ln->tr_C == M, "linear_16: LayerNorm transpose shape %d x %d != %lld rows",
                   ln->tr_R, ln->tr_C, M);
    g.ln_w = ln->w; g.ln_b = ln->b; g.ln_out = ln->out; g.ln_eps = ln->eps; g.ln_fp16 = ln->out_fp16;
    g.ln_tr_R = ln->tr_R; g.ln_tr_C = ln->tr_C; g.ln_counters = ln->counters;
    {
      const char* e = getenv("RNAMSM_LN_DEBUG");
      g.ln_debug = e ? atoi(e) : 0;
    }
    return launch_variant<V_DENSE, BLOCK_N, true>(ta, tb, to, g, linear_class(epi.kind, N, K), st);
  }
  static int wide = -1;                      // RNAMSM_GELU_WIDE=0: the 8-warp epilogue for the GELU instance too (A/B runs)
  if (wide < 0) { const char* e = getenv("RNAMSM_GELU_WIDE"); wide = (e && e[0] == '0') ? 0 : 1; }
  if (epi.kind == RNAMSM_EPI_BIAS_GELU && wide)
    return launch_variant<V_DENSE, BLOCK_N, false, false, true>(ta, tb, to, g, linear_class(epi.kind, N, K), st);
  return launch_variant<V_DENSE>(ta, tb, to, g, linear_class(epi.kind, N, K), st);
}

// fp32 nn.Linear on the tensor cores: x = x_hi + x_lo, W = W_hi + W_lo (split_tf32 in elementwise.cu), three tf32 MMAs per
// k-step.  out: fp32 [M, N] (bias / bias+GELU epilogues: plain store; residual epilogue: reduce-add in place).
int launch_linear_tf32(const float* x_hi, const float* x_lo, const float* W_hi, const float* W_lo, long long M, int N, int K,
                       const LinearEpilogue& epi, float* out, cudaStream_t st) {
  RNAMSM_REQUIRE(M > 0 && M < (1LL << 31), "linear_tf32: M=%lld out of range", M);
  RNAMSM_REQUIRE(N % 32 == 0 && K % 32 == 0 && K >= 32, "linear_tf32: N=%d and K=%d must be multiples of 32", N, K);
  RNAMSM_REQUIRE(epi.bias != nullptr && epi.q_cols % 64 == 0, "linear_tf32: bias required, q_cols a multiple of 64");
  CUtensorMap ta, tb, to;
  PeerMaps lo{};
  uint64_t adims[3] = {(uint64_t)K, (uint64_t)M, 1}, astr[2] = {(uint64_t)K * 4, (uint64_t)M * K * 4};
  uint64_t bdims[3] = {(uint64_t)K, (uint64_t)N, 1}, bstr[2] = {(uint64_t)K * 4, (uint64_t)N * K * 4};
  uint32_t abox[3] = {32, BLOCK_M, 1}, bbox[3] = {32, HALF_N, 1};
  if (encode_tmap(&ta, TMAP_F32, x_hi, 3, adims, astr, abox)) return 3;
  if (encode_tmap(&lo.m[0], TMAP_F32, x_lo, 3, adims, astr, abox)) return 3;
  if (encode_tmap(&tb, TMAP_F32, W_hi, 3, bdims, bstr, bbox)) return 3;
  if (encode_tmap(&lo.m[1], TMAP_F32, W_lo, 3, bdims, bstr, bbox)) return 3;
  uint64_t odims[3] = {(uint64_t)N, (uint64_t)M, 1}, ostr[2] = {(uint64_t)N * 4, (uint64_t)M * N * 4};
  uint32_t obox[3] = {32, 32, 1};
  if (encode_tmap(&to, TMAP_F32, out, 3, odims, ostr, obox)) return 3;
  GemmArgs g{};
  g.m_tiles = ceil_div(M, PAIR_M);
  g.n_tiles = ceil_div(N, BLOCK_N);
  g.batches = 1; g.splits = 1;
  g.k_blocks = K / 32;
  g.M = (int)M; g.N = N;
  g.epi_kind = epi.kind; g.bias = epi.bias; g.q_scale = epi.q_scale; g.q_cols = epi.q_cols; g.row_mask = epi.row_mask;
  g.out = out; g.ld_out = N;
  return launch_variant<V_DENSE, BLOCK_N, false, true>(ta, tb, to, g, linear_class(epi.kind, N, K), st, &lo);
}

// Column block's out-projection of the sharded forward: ctx [R*Cn, K] (this rank's column shard, token-major
// (r, c_local)) x W[N, K]^T + bias, reduce-added into the row owners' residual streams (peer_x[g]: fp32
// [Rn*C, N] on rank g).
int launch_linear_16_scatter(const void* x, const void* W, const float* bias, int R, int Cn, int N, int K, int fp16,
                             void* const* peer_x, int n_ranks, int Rn, int C, int c0, int as_delta16, cudaStream_t st) {
  const long long M = (long long)R * Cn;
  RNAMSM_REQUIRE(M > 0 && M < (1LL << 31), "linear_scatter: M=%lld out of range", M);
  RNAMSM_REQUIRE(N % 64 == 0 && K % BLOCK_K == 0 && K >= BLOCK_K, "linear_scatter: N=%d and K=%d must be multiples of 64", N, K);
  RNAMSM_REQUIRE(n_ranks >= 1 && n_ranks <= RNAMSM_MAX_PEERS && Rn * n_ranks == R, "linear_scatter: R=%d != %d ranks x Rn=%d", R, n_ranks, Rn);
  RNAMSM_REQUIRE(Cn % 16 == 0, "linear_scatter: columns per rank Cn=%d must be a multiple of 16 (TMA box rows)", Cn);
  // the shard is the (c0 / Cn)-th of n_ranks inside the owners' C columns (m_tile_shift relies on c0 / Cn < n_ranks)
  RNAMSM_REQUIRE(Cn > 0 && c0 >= 0 && c0 % Cn == 0 && c0 + Cn <= C && c0 / Cn < n_ranks,
                 "linear_scatter: column shard [%d, %d + %d) is not one of %d shards of C=%d", c0, c0, Cn, n_ranks, C);
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  const int box_rows = Cn % 32 == 0 ? 32 : 16;
  CUtensorMap ta, tb;
  PeerMaps pm{};
  {
    uint64_t dims[3] = {(uint64_t)K, (uint64_t)M, 1};
    uint64_t strides[2] = {(uint64_t)K * 2, (uint64_t)M * K * 2};
    uint32_t box[3] = {BLOCK_K, BLOCK_M, 1};
    if (encode_tmap(&ta, in_dt, x, 3, dims, strides, box)) return 3;
  }
  {
    uint64_t dims[3] = {(uint64_t)K, (uint64_t)N, 1};
    uint64_t strides[2] = {(uint64_t)K * 2, (uint64_t)N * K * 2};
    uint32_t box[3] = {BLOCK_K, HALF_N, 1};
    if (encode_tmap(&tb, in_dt, W, 3, dims, strides, box)) return 3;
  }
  for (int g = 0; g < n_ranks; ++g) {       // peer_x[g]: fp32 residual [Rn*C, N], or 16-bit receive buffer of the same shape
    const uint64_t el = as_delta16 ? 2 : 4;
    uint64_t dims[3] = {(uint64_t)N, (uint64_t)C, (uint64_t)Rn};
    uint64_t strides[2] = {(uint64_t)N * el, (uint64_t)C * N * el};
    uint32_t box[3] = {as_delta16 ? 64u : 32u, (uint32_t)box_rows, 1};
    if (encode_tmap(&pm.m[g], as_delta16 ? in_dt : TMAP_F32, peer_x[g], 3, dims, strides, box)) return 3;
  }
  GemmArgs g{};
  g.m_tiles = ceil_div(M, PAIR_M);
  g.n_tiles = ceil_div(N, BLOCK_N);
  g.batches = 1; g.splits = 1;
  g.k_blocks = K / BLOCK_K;
  g.M = (int)M; g.N = N;
  g.fp16 = fp16;
  g.epi_kind = as_delta16 ? RNAMSM_EPI_BIAS : RNAMSM_EPI_BIAS_RESIDUAL; g.bias = bias; g.q_scale = 1.f;
  g.peer_n = n_ranks; g.peer_Rn = Rn; g.peer_Cn = Cn; g.peer_c0 = c0; g.peer_box_rows = box_rows;
  g.m_tile_shift = (int)(((long long)(c0 / Cn) * g.m_tiles) / n_ranks);   // rank * m_tiles / n: start at our own rows' owner
  return launch_variant<V_DENSE>(ta, tb, pm.m[0], g, KC_LINEAR_OUT, st, &pm);
}

int gemm_max_pairs() { ensure_max_pairs(); return g_max_pairs; }

static inline int tied_tile_n(int C) { return C <= 64 ? 64 : (C <= 128 ? 128 : BLOCK_N); }

int row_logits_splits_16(int R, int C, int H) {
  const long long tiles = (long long)H * ceil_div(C, PAIR_M) * ceil_div(C, tied_tile_n(C));
  ensure_max_pairs();
  const int pairs = g_max_pairs;
  // fewer tiles than pairs: the LARGEST split count that still fits one wave (12 head tiles x 6 splits = 72 of 74
  // pairs; rounding up to 7 would spill 10 tiles into a second, almost empty wave and double the time)
  int want = (int)std::max<long long>(1, pairs / tiles);
  if (tiles > pairs) {
    // more tiles than pairs: pick the split count in [1, 4] with the best wave efficiency
    double best = 0.0;
    want = 1;
    for (int s = 1; s <= 4; ++s) {
      const long long tt = tiles * s;
      const double eff = (double)tt / ((double)((tt + pairs - 1) / pairs) * pairs);
      if (eff > best + 0.03) { best = eff; want = s; }
    }
  }
  want = std::min(want, std::max(1, R / 8));  // keep >= 8 rows (k-blocks) per split
  want = std::max(1, std::min(want, R));
  const int rps = ceil_div(R, want);
  return ceil_div(R, rps);  // every split non-empty
}

int launch_row_logits_16(const void* qkv, int R, int C, int H, int fp16, float* partial, int n_splits, cudaStream_t st) {
  RNAMSM_REQUIRE(n_splits >= 1 && n_splits <= R, "row_logits_16: n_splits=%d out of range for R=%d", n_splits, R);
  const int rps = ceil_div(R, n_splits);
  RNAMSM_REQUIRE((n_splits - 1) * rps < R, "row_logits_16: n_splits=%d leaves an empty split for R=%d", n_splits, R);
  const int ld = 3 * H * 64;
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  CUtensorMap ta, tb;
  uint64_t dims[3] = {(uint64_t)ld, (uint64_t)C, (uint64_t)R};
  uint64_t strides[2] = {(uint64_t)ld * 2, (uint64_t)C * ld * 2};
  const int bn = tied_tile_n(C);
  uint32_t box_a[3] = {BLOCK_K, BLOCK_M, 1};
  uint32_t box_b[3] = {BLOCK_K, (uint32_t)(bn / 2), 1};
  if (encode_tmap(&ta, in_dt, qkv, 3, dims, strides, box_a)) return 3;
  if (encode_tmap(&tb, in_dt, qkv, 3, dims, strides, box_b)) return 3;
  GemmArgs g{};
  g.m_tiles = ceil_div(C, PAIR_M);
  g.n_tiles = ceil_div(C, bn);
  g.batches = H; g.splits = n_splits;
  g.rows_per_split = rps;
  g.R = R; g.C = C; g.H = H; g.M = C; g.N = C;
  g.fp16 = fp16;
  g.out = partial;
  if (bn == 64) return launch_variant<V_TIED, 64>(ta, tb, ta, g, KC_ROW_LOGITS, st);
  if (bn == 128) return launch_variant<V_TIED, 128>(ta, tb, ta, g, KC_ROW_LOGITS, st);
  return launch_variant<V_TIED>(ta, tb, ta, g, KC_ROW_LOGITS, st);
}

int launch_row_av_16(const void* probs, int ldp, const void* qkv, int R, int C, int H, int fp16, void* ctx,
                     cudaStream_t st) {
  RNAMSM_REQUIRE(ldp % 8 == 0 && ldp >= C, "row_av_16: ldp=%d must be a multiple of 8 and >= C=%d", ldp, C);
  const int ld = 3 * H * 64;
  const int in_dt = fp16 ? TMAP_F16 : TMAP_BF16;
  CUtensorMap ta, tb, to;
  {
    uint64_t dims[3] = {(uint64_t)C, (uint64_t)C, (uint64_t)H};
    uint64_t strides[2] = {(uint64_t)ldp * 2, (uint64_t)C * ldp * 2};
    uint32_t box[3] = {BLOCK_K, BLOCK_M, 1};
    if (encode_tmap(&ta, in_dt, probs, 3, dims, strides, box)) return 3;
  }
  {
    uint64_t dims[3] = {(uint64_t)ld, (uint64_t)C, (uint64_t)R};
    uint64_t strides[2] = {(uint64_t)ld * 2, (uint64_t)C * ld * 2};
    uint32_t box[3] = {64, BLOCK_K, 2};
    if (encode_tmap(&tb, in_dt, qkv, 3, dims, strides, box)) return 3;
  }
  {
    uint64_t dims[3] = {(uint64_t)(H * 64), (uint64_t)C, (uint64_t)R};
    uint64_t strides[2] = {(uint64_t)H * 64 * 2, (uint64_t)C * H * 64 * 2};
    uint32_t box[3] = {64, 32, 1};
    if (encode_tmap(&to, in_dt, ctx, 3, dims, strides, box)) return 3;
  }
  GemmArgs g{};
  g.m_tiles = ceil_div(C, PAIR_M);
  g.n_tiles = ceil_div(R, 4);
  g.batches = H; g.splits = 1;
  g.k_blocks = ceil_div(C, BLOCK_K);
  g.R = R; g.C = C; g.H = H; g.M = C; g.N = R;
  g.fp16 = fp16;
  g.out = ctx; g.ld_out = H * 64;
  // the A V tile has K = C: at C = 256 only four k-blocks of MMAs stand against a 256 x 256 16-bit epilogue, so the
  // 16-warp epilogue (kWide, see above) is what bounds the tile less
  static int wide = -1;
  if (wide < 0) { const char* e = getenv("RNAMSM_AV_WIDE"); wide = (e && e[0] == '0') ? 0 : 1; }
  if (wide) return launch_variant<V_AV, BLOCK_N, false, false, true>(ta, tb, to, g, KC_ROW_AV, st);
  return launch_variant<V_AV>(ta, tb, to, g, KC_ROW_AV, st);
}

}  // namespace rnamsm
