// Peer-memory plumbing and the fused compute + exchange kernels of the sharded single-MSA forward
// (SURVEY.md 8e; rna-msm_b200/sharded.py).  One process per GPU; buffers that other GPUs touch are
// cudaMalloc'ed here, exported as CUDA IPC handles (exchanged by the host over torch.distributed) and
// mapped into every peer, so kernels read / write them directly over NVLink:
//
//   layernorm_push_kernel   LayerNorm of the row shard, each 16-bit output row stored straight into
//                           the COLUMN OWNER's buffer in its final [C/n, R, D] order: the row->column
//                           all-to-all costs no extra pass and no NCCL call
//   row_softmax_p2p_kernel  the tied-logit exchange: every rank owns C/n query rows, PULLS the partial
//                           logits of those rows from all ranks (reduce-scatter), applies scale / key
//                           mask / softmax, and PUSHES the 16-bit probabilities to all ranks (all-gather);
//                           the fp32 map rows stay in the owner's `map_out` (every rank copies its own rows
//                           to the host over its own PCIe link) -- one kernel instead of all-reduce +
//                           softmax, moving (n-1)/n^2 of the logits in and the 16-bit rows out
//   (umma_gemm.cu)          the column block's out-projection reduces its result into the ROW OWNER's
//                           fp32 residual stream with TMA reduce-add on peer tensor maps: GEMM, the
//                           column->row all-to-all and the residual add in one kernel
//
// Ordering between GPUs: peer_barrier_kernel, a flag barrier in peer memory launched on the stream between phases.
#include <cuda_fp16.h>
#include <string.h>

#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

struct PeerPtrs { void* p[RNAMSM_MAX_PEERS]; };

constexpr int kMaxVecP = 8;
constexpr int kLnWarpsP = 8;

// kOut: 1 = bf16, 2 = fp16.  Input row (r_local, c) of the row shard -> peer d = c / Cn, output row
// (c - d*Cn) * R + (r0 + r_local)   [column-major token order of the column shard].
template <int kOut>
__global__ void __launch_bounds__(kLnWarpsP * 32)
layernorm_push_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                      PeerPtrs dst, int Rn, int C, int Cn, int R, int r0, int D, float eps, int c_shift) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nv = D / 128;
  const long long n_rows = (long long)Rn * C;
  for (long long it = (long long)blockIdx.x * kLnWarpsP + warp; it < n_rows; it += (long long)gridDim.x * kLnWarpsP) {
    // every rank walks the columns starting at its own shard (c_shift), so at any moment the ranks
    // write to DIFFERENT column owners instead of all hitting the same one's NVLink ingress
    const int r_it = (int)(it / C);
    int c_it = (int)(it % C) + c_shift;
    if (c_it >= C) c_it -= C;
    const long long row = (long long)r_it * C + c_it;
    const float* src = x + (size_t)row * D;
    float4 v[kMaxVecP];
#pragma unroll
    for (int i = 0; i < kMaxVecP; ++i)
      if (i < nv) v[i] = *reinterpret_cast<const float4*>(src + lane * 4 + i * 128);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxVecP; ++i)
      if (i < nv) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxVecP; ++i)
      if (i < nv) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
      }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
    const int r_local = (int)(row / C), c = (int)(row % C);
    const int d = c / Cn;
    uint16_t* out = reinterpret_cast<uint16_t*>(dst.p[d]) + ((size_t)(c - d * Cn) * R + r0 + r_local) * D;
#pragma unroll
    for (int i = 0; i < kMaxVecP; ++i)
      if (i < nv) {
        const int f = lane * 4 + i * 128;
        const float4 ww = *reinterpret_cast<const float4*>(w + f);
        const float4 bb = *reinterpret_cast<const float4*>(b + f);
        const float y0 = v[i].x * rstd * ww.x + bb.x, y1 = v[i].y * rstd * ww.y + bb.y;
        const float y2 = v[i].z * rstd * ww.z + bb.z, y3 = v[i].w * rstd * ww.w + bb.w;
        const uint2 pk = kOut == 1 ? make_uint2(pack_bf16(y0, y1), pack_bf16(y2, y3))
                                   : make_uint2(pack_f16(y0, y1), pack_f16(y2, y3));
        *reinterpret_cast<uint2*>(out + f) = pk;
      }
  }
}

// One warp per (head, owned query row i).  partial slabs: [n_splits, H, C, C] fp32 on every rank.
template <int kLp>
__global__ void __launch_bounds__(128)
row_softmax_p2p_kernel(PeerPtrs partial, int n_ranks, int rank, int n_splits, int H, int C, int i0, int i1,
                       const uint8_t* __restrict__ key_pad, float logit_scale, float* map_out, PeerPtrs probs,
                       int ld_lp) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rows_owned = i1 - i0;
  const long long idx = (long long)blockIdx.x * 4 + warp;            // h * rows_owned + (i - i0)
  if (idx >= (long long)H * rows_owned) return;
  const int h = (int)(idx / rows_owned), i = i0 + (int)(idx % rows_owned);
  const size_t row_off = ((size_t)h * C + i) * C;
  const size_t split_stride = (size_t)H * C * C;
  auto logit = [&](int j) -> float {
    float a = 0.f;
    for (int t = 1; t <= n_ranks; ++t) {            // start at the next rank: no two ranks pull from the same source at once
      const float* src = reinterpret_cast<const float*>(partial.p[(rank + t) % n_ranks]) + row_off;
      for (int s = 0; s < n_splits; ++s) a += src[s * split_stride + j];
    }
    a *= logit_scale;
    if (key_pad && key_pad[j]) a = -10000.f;                          // masked_fill, modules.py:780-784
    return a;
  };
  // the summed row lives in registers when it fits (C <= 1024): one pass over the remote data
  constexpr int kMaxPerLane = 32;
  float vals[kMaxPerLane];
  const bool cached = C <= 32 * kMaxPerLane;
  float mx = -INFINITY;
  if (cached) {
#pragma unroll
    for (int t = 0; t < kMaxPerLane; ++t) {
      const int j = lane + 32 * t;
      vals[t] = j < C ? logit(j) : -INFINITY;
      mx = fmaxf(mx, vals[t]);
    }
  } else {
    for (int j = lane; j < C; j += 32) mx = fmaxf(mx, logit(j));
  }
  mx = warp_max(mx);
  float sum = 0.f;
  if (cached) {
#pragma unroll
    for (int t = 0; t < kMaxPerLane; ++t) {
      vals[t] = (lane + 32 * t < C) ? __expf(vals[t] - mx) : 0.f;
      sum += vals[t];
    }
  } else {
    for (int j = lane; j < C; j += 32) sum += __expf(logit(j) - mx);
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  float* mdst = map_out ? map_out + row_off : nullptr;
  const size_t lp_off = ((size_t)h * C + i) * ld_lp;
  auto emit = [&](int j, float p) {                 // fp32 map row -> map_out (local); 16-bit row -> every rank
    if (mdst && j < C) mdst[j] = p;
    if (j < ld_lp) {
      for (int t = 0; t < n_ranks; ++t) {
        const int g = (rank + t) % n_ranks;
        if constexpr (kLp == 1)
          reinterpret_cast<__nv_bfloat16*>(probs.p[g])[lp_off + j] = __float2bfloat16(p);
        else
          reinterpret_cast<__half*>(probs.p[g])[lp_off + j] = __float2half_rn(p);
      }
    }
  };
  if (cached) {
#pragma unroll
    for (int t = 0; t < kMaxPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < ld_lp || j < C) emit(j, j < C ? vals[t] * inv : 0.f);
    }
    for (int j = 32 * kMaxPerLane + lane; j < ld_lp; j += 32) emit(j, 0.f);   // (ld_lp may exceed 32 kMaxPerLane)
  } else {
    for (int j = lane; j < ld_lp || j < C; j += 32) emit(j, j < C ? __expf(logit(j) - mx) * inv : 0.f);
  }
}

// Block-per-row, 128-bit version for C % 4 == 0 (every production shape): 128 threads own one (head,
// query row), thread t holds columns 4t + 512k.  All remote float4 loads of a row are issued before
// the first use (NVLink latency ~2 us), the fp32 map row leaves as float4 stores to map_out, the 16-bit
// row as 8-byte stores to every rank.
constexpr int kP2pT = 8;   // C <= 512 * kP2pT

template <int kLp>
__global__ void __launch_bounds__(128)
row_softmax_p2p_vec_kernel(PeerPtrs partial, int n_ranks, int rank, int n_splits, int H, int C, int i0, int rows_owned,
                           const uint8_t* __restrict__ key_pad, float logit_scale, float* map_out, PeerPtrs probs,
                           int ld_lp) {
  __shared__ float red[8];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int h = blockIdx.x / rows_owned, i = i0 + blockIdx.x % rows_owned;
  const size_t row_off = ((size_t)h * C + i) * C;
  const size_t split_stride = (size_t)H * C * C;
  float acc[kP2pT][4];
#pragma unroll
  for (int k = 0; k < kP2pT; ++k)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[k][e] = 0.f;
  for (int t = 1; t <= n_ranks; ++t) {              // rotated: rank r pulls from r+1, r+2, ... (no source hot spot)
    const float* src = reinterpret_cast<const float*>(partial.p[(rank + t) % n_ranks]) + row_off;
    for (int s = 0; s < n_splits; ++s) {
#pragma unroll
      for (int k = 0; k < kP2pT; ++k) {
        const int j = 4 * tid + 512 * k;
        if (j < C) {
          const float4 v = *reinterpret_cast<const float4*>(src + s * split_stride + j);
          acc[k][0] += v.x; acc[k][1] += v.y; acc[k][2] += v.z; acc[k][3] += v.w;
        }
      }
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < kP2pT; ++k) {
    const int j = 4 * tid + 512 * k;
    if (j < C) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float a = acc[k][e] * logit_scale;
        if (key_pad && key_pad[j + e]) a = -10000.f;                  // masked_fill, modules.py:780-784
        acc[k][e] = a;
        mx = fmaxf(mx, a);
      }
    }
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < kP2pT; ++k) {
    const int j = 4 * tid + 512 * k;
    if (j < C) {
#pragma unroll
      for (int e = 0; e < 4; ++e) { acc[k][e] = __expf(acc[k][e] - mx); sum += acc[k][e]; }
    }
  }
  sum = warp_sum(sum);
  if (lane == 0) red[4 + warp] = sum;
  __syncthreads();
  const float inv = 1.f / ((red[4] + red[5]) + (red[6] + red[7]));
  const size_t lp_off = ((size_t)h * C + i) * ld_lp;
#pragma unroll
  for (int k = 0; k < kP2pT; ++k) {
    const int j = 4 * tid + 512 * k;
    if (j < C) {
      const float4 p = make_float4(acc[k][0] * inv, acc[k][1] * inv, acc[k][2] * inv, acc[k][3] * inv);
      if (map_out) *reinterpret_cast<float4*>(map_out + row_off + j) = p;
      const uint2 pk = kLp == 1 ? make_uint2(pack_bf16(p.x, p.y), pack_bf16(p.z, p.w))
                                : make_uint2(pack_f16(p.x, p.y), pack_f16(p.z, p.w));
      for (int t = 0; t < n_ranks; ++t)
        *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(probs.p[(rank + t) % n_ranks]) + lp_off + j) = pk;
    } else if (j < ld_lp) {                                           // zero the padding columns [C, ld_lp)
      for (int t = 0; t < n_ranks; ++t)
        *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(probs.p[(rank + t) % n_ranks]) + lp_off + j) = make_uint2(0u, 0u);
    }
  }
  for (int j = 512 * kP2pT + 4 * tid; j < ld_lp; j += 512)            // padding past column 512 kP2pT (C = 4096 < ld_lp)
    for (int t = 0; t < n_ranks; ++t)
      *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(probs.p[(rank + t) % n_ranks]) + lp_off + j) = make_uint2(0u, 0u);
}


// -------------------------------------------------------------------------------------------
// Cross-GPU barrier on the stream, in peer memory (replaces a host-launched 4-byte NCCL all-reduce per phase).
// Every rank owns a flag array `flags[n]` (peer-mapped); rank r arrives by storing the barrier's epoch into
// slot r of EVERY rank's array (st.release.sys over NVLink) and leaves once its own n slots have all reached the
// epoch (ld.acquire.sys).  Kernels launched before it on the stream have completed (stream order), so their
// peer writes are performed before the release; kernels after it start only once every peer has arrived.
// Epochs only grow, so a peer that is already one barrier ahead still satisfies the wait.  The wait is bounded:
// a rank that never arrives traps instead of hanging the box.
// -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
peer_barrier_kernel(PeerPtrs flags, int n_ranks, int rank, unsigned epoch) {
  const int t = threadIdx.x;
  if (t < n_ranks) {
    __threadfence_system();
    unsigned* remote = reinterpret_cast<unsigned*>(flags.p[t]) + rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(remote), "r"(epoch) : "memory");
    const unsigned* mine = reinterpret_cast<const unsigned*>(flags.p[rank]) + t;
    unsigned v = 0;
    long long spins = 0;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if ((int)(v - epoch) >= 0) break;
      __nanosleep(200);
      if (++spins > (1LL << 25)) {      // ~10 s
        printf("rnamsm: peer barrier timeout (rank %d waiting for rank %d, epoch %u, saw %u)\n", rank, t, epoch, v);
        __trap();
      }
    }
  }
  __syncwarp();
  __threadfence_system();
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

int rnamsm_peer_alloc(size_t bytes, void** out) {
  RNAMSM_REQUIRE(out != nullptr && bytes > 0, "peer_alloc: bad arguments");
  RNAMSM_CHECK_CUDA(cudaMalloc(out, bytes));
  RNAMSM_CHECK_CUDA(cudaMemset(*out, 0, bytes));
  return 0;
}
int rnamsm_peer_free(void* p) {
  if (p) RNAMSM_CHECK_CUDA(cudaFree(p));
  return 0;
}
int rnamsm_ipc_export(const void* p, void* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  RNAMSM_CHECK_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), const_cast<void*>(p)));
  return 0;
}
int rnamsm_ipc_import(const void* handle64, void** out) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  RNAMSM_CHECK_CUDA(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
int rnamsm_ipc_close(void* p) {
  if (p) RNAMSM_CHECK_CUDA(cudaIpcCloseMemHandle(p));
  return 0;
}

int rnamsm_layernorm_push(const float* x, const float* w, const float* b, void* const* peer_dst, int n_ranks, int Rn,
                          int C, int R, int r0, int D, float eps, int y_dtype, void* stream) {
  RNAMSM_REQUIRE(n_ranks >= 1 && n_ranks <= RNAMSM_MAX_PEERS, "layernorm_push: %d ranks (max %d)", n_ranks, RNAMSM_MAX_PEERS);
  RNAMSM_REQUIRE(C % n_ranks == 0 && D % 128 == 0 && D <= 1024, "layernorm_push: C=%d must divide by %d ranks; D=%d", C, n_ranks, D);
  RNAMSM_REQUIRE(y_dtype == RNAMSM_BF16 || y_dtype == RNAMSM_F16, "layernorm_push: 16-bit output only");
  RNAMSM_REQUIRE(Rn >= 0 && r0 >= 0 && r0 + Rn <= R, "layernorm_push: rows [%d, %d + %d) outside the R=%d rows of the MSA", r0, r0, Rn, R);
  PeerPtrs dst{};
  for (int g = 0; g < n_ranks; ++g) dst.p[g] = peer_dst[g];
  const long long n_rows = (long long)Rn * C;
  if (n_rows <= 0) return 0;
  const int blocks = (int)std::min<long long>((n_rows + kLnWarpsP - 1) / kLnWarpsP, 148LL * 32);
  cudaStream_t st = (cudaStream_t)stream;
  const int c_shift = (int)(((long long)(r0 / (Rn > 0 ? Rn : 1)) * (C / n_ranks)) % C);   // = rank * Cn
  ProfScope prof(KC_LAYERNORM, st);
  if (y_dtype == RNAMSM_BF16)
    layernorm_push_kernel<1><<<blocks, kLnWarpsP * 32, 0, st>>>(x, w, b, dst, Rn, C, C / n_ranks, R, r0, D, eps, c_shift);
  else
    layernorm_push_kernel<2><<<blocks, kLnWarpsP * 32, 0, st>>>(x, w, b, dst, Rn, C, C / n_ranks, R, r0, D, eps, c_shift);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int rnamsm_linear_residual_scatter(const void* ctx, const void* W, const float* bias, int R, int Cn, int N, int K,
                                   int dtype, void* const* peer_x, int n_ranks, int Rn, int C, int c0, int as_delta16,
                                   void* stream) {
  RNAMSM_REQUIRE(dtype == RNAMSM_BF16 || dtype == RNAMSM_F16, "linear_residual_scatter: 16-bit operands only");
  return launch_linear_16_scatter(ctx, W, bias, R, Cn, N, K, dtype == RNAMSM_F16, peer_x, n_ranks, Rn, C, c0, as_delta16,
                                  (cudaStream_t)stream);
}

int rnamsm_add_layernorm(float* x, const void* delta, int delta_dtype, const float* w, const float* b, void* y,
                         int y_dtype, long long n_rows, int D, float eps, void* stream) {
  return launch_add_layernorm(x, delta, delta_dtype, w, b, y, y_dtype, n_rows, D, eps, (cudaStream_t)stream);
}

int rnamsm_row_softmax_p2p(void* const* peer_partial, int n_ranks, int rank, int n_splits, int H, int C,
                           const uint8_t* key_pad, float logit_scale, float* map_out, void* const* peer_probs,
                           int ld_lp, int dtype, void* stream) {
  RNAMSM_REQUIRE(n_ranks >= 1 && n_ranks <= RNAMSM_MAX_PEERS && rank >= 0 && rank < n_ranks, "row_softmax_p2p: bad rank %d/%d", rank, n_ranks);
  RNAMSM_REQUIRE(C % n_ranks == 0, "row_softmax_p2p: C=%d must divide by %d ranks", C, n_ranks);
  RNAMSM_REQUIRE(dtype == RNAMSM_BF16 || dtype == RNAMSM_F16, "row_softmax_p2p: 16-bit probabilities only");
  PeerPtrs pp{}, pr{};
  for (int g = 0; g < n_ranks; ++g) { pp.p[g] = peer_partial[g]; pr.p[g] = peer_probs[g]; }
  const int Cq = C / n_ranks, i0 = rank * Cq, i1 = i0 + Cq;
  const long long rows = (long long)H * Cq;
  const int blocks = (int)((rows + 3) / 4);
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof(KC_ROW_SOFTMAX, st);
  if (C % 4 == 0 && C <= 512 * kP2pT && ld_lp % 4 == 0) {
    if (dtype == RNAMSM_BF16)
      row_softmax_p2p_vec_kernel<1><<<(int)rows, 128, 0, st>>>(pp, n_ranks, rank, n_splits, H, C, i0, Cq, key_pad, logit_scale,
                                                            map_out, pr, ld_lp);
    else
      row_softmax_p2p_vec_kernel<2><<<(int)rows, 128, 0, st>>>(pp, n_ranks, rank, n_splits, H, C, i0, Cq, key_pad, logit_scale,
                                                            map_out, pr, ld_lp);
    count_launch();
    RNAMSM_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  if (dtype == RNAMSM_BF16)
    row_softmax_p2p_kernel<1><<<blocks, 128, 0, st>>>(pp, n_ranks, rank, n_splits, H, C, i0, i1, key_pad, logit_scale, map_out, pr, ld_lp);
  else
    row_softmax_p2p_kernel<2><<<blocks, 128, 0, st>>>(pp, n_ranks, rank, n_splits, H, C, i0, i1, key_pad, logit_scale, map_out, pr, ld_lp);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}


int rnamsm_peer_barrier(void* const* peer_flags, int n_ranks, int rank, unsigned int epoch, void* stream) {
  RNAMSM_REQUIRE(n_ranks >= 1 && n_ranks <= RNAMSM_MAX_PEERS && rank >= 0 && rank < n_ranks, "peer_barrier: bad rank %d/%d", rank, n_ranks);
  PeerPtrs f{};
  for (int g = 0; g < n_ranks; ++g) {
    RNAMSM_REQUIRE(peer_flags[g] != nullptr, "peer_barrier: null flag array for rank %d", g);
    f.p[g] = peer_flags[g];
  }
  peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, n_ranks, rank, epoch);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// Query rows [i0, i1) of one layer's maps [H, C, C] (device) -> the BOS/EOS-stripped host layout [H, Ls, Ls]
// (RNA_MSM_Inference.py:150-158: attentions[..., start:end, start:end]) in ONE pitched DMA.  Each rank of the sharded
// forward copies only the rows it owns, over its own PCIe link, into a host buffer shared by the ranks.
int rnamsm_copy_map_rows_d2h(const float* maps_layer, int H, int C, int i0, int i1, int start, int Ls, float* host_layer,
                             void* stream) {
  RNAMSM_REQUIRE(H > 0 && C > 0 && start >= 0 && Ls > 0 && start + Ls <= C, "copy_map_rows_d2h: bad shape C=%d start=%d Ls=%d", C, start, Ls);
  const int lo = i0 > start ? i0 : start, hi = i1 < start + Ls ? i1 : start + Ls;
  if (hi <= lo) return 0;
  cudaMemcpy3DParms p;
  memset(&p, 0, sizeof(p));
  p.srcPtr = make_cudaPitchedPtr(const_cast<float*>(maps_layer), (size_t)C * 4, (size_t)C * 4, (size_t)C);
  p.srcPos = make_cudaPos((size_t)start * 4, (size_t)lo, 0);
  p.dstPtr = make_cudaPitchedPtr(host_layer, (size_t)Ls * 4, (size_t)Ls * 4, (size_t)Ls);
  p.dstPos = make_cudaPos(0, (size_t)(lo - start), 0);
  p.extent = make_cudaExtent((size_t)Ls * 4, (size_t)(hi - lo), (size_t)H);
  p.kind = cudaMemcpyDeviceToHost;
  RNAMSM_CHECK_CUDA(cudaMemcpy3DAsync(&p, (cudaStream_t)stream));
  return 0;
}

int rnamsm_host_register(void* p, size_t bytes) {
  RNAMSM_REQUIRE(p != nullptr && bytes > 0, "host_register: bad arguments");
  RNAMSM_CHECK_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  return 0;
}
int rnamsm_host_unregister(void* p) {
  if (p) RNAMSM_CHECK_CUDA(cudaHostUnregister(p));
  return 0;
}

}  // extern "C"
