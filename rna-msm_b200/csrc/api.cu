// C ABI of librnamsm_b200.so (declared in include/rnamsm_b200.h) and the host-side drivers that
// chain the kernels into one AxialTransformerLayer (modules.py:242-267) / one MSATransformer
// forward (model.py:338-416).  No allocation, no synchronisation: everything is enqueued on the
// caller's stream against caller-owned buffers.
#include <cudaTypedefs.h>
#include <stdarg.h>
#include <stdlib.h>

#include <atomic>
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---- optional kernel-class timing ---------------------------------------------------------------
struct ProfEvent { int cls; cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::vector<ProfEvent> g_prof_events;
static std::vector<cudaEvent_t> g_prof_pool;
static const char* kClassNames[KC_COUNT] = {"embed_ln", "layernorm", "row_softmax", "vocab_proj", "linear_qkv",
                                            "linear_fc1_gelu", "linear_out_resid", "linear_fc2_resid",
                                            "row_logits", "row_av", "col_attn", "contact_head", "row_attn_short",
                                            "window_build", "window_stitch"};
static cudaEvent_t prof_get_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
ProfScope::ProfScope(int c, cudaStream_t s) : cls(c), st(s), slot(nullptr) {
  if (!g_prof_on) return;
  ProfEvent ev{c, prof_get_event(), prof_get_event()};
  cudaEventRecord(ev.a, st);
  g_prof_events.push_back(ev);
  slot = reinterpret_cast<void*>(g_prof_events.size());
}
ProfScope::~ProfScope() {
  if (!slot) return;
  cudaEventRecord(g_prof_events[reinterpret_cast<size_t>(slot) - 1].b, st);
}

// RNAMSM_PDL=1 launches the forward's kernels with programmatic dependent launch (each kernel's prologue overlaps its
// predecessor's tail; all parity tests pass with it).  OFF by default: measured no gain on a B200 -- 512 x 36 (132
// launches of ~40 us): 5.358 ms plain vs 5.352 ms; 512 x 256: within the box-to-box clock noise -- back-to-back launches
// on one stream already pipeline, and a persistent 230 KiB CTA cannot become resident before its predecessor's CTA on
// that SM has exited.
bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RNAMSM_PDL");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

int encode_tmap(CUtensorMap* map, int elem, const void* base, int rank, const uint64_t* dims,
                const uint64_t* strides_bytes, const uint32_t* box) {
  static PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled entry point unavailable (%s)", cudaGetErrorString(e));
      return 1;
    }
    encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_error("TMA base pointer %p is not 16-byte aligned", base);
    return 1;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    estr[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_bytes[i - 1];
      if (gstr[i - 1] % 16 != 0) {
        set_error("TMA stride %llu (dim %d) is not a multiple of 16 bytes", (unsigned long long)gstr[i - 1], i);
        return 1;
      }
    }
  }
  const CUtensorMapDataType dt = elem == TMAP_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : elem == TMAP_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = encode(map, dt, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx,
                      estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu,%llu box %u,%u,%u)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
    return 1;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Workspace plan for one R x C MSA (bytes, every region 256 B aligned):
//   xn      [T, D]      compute dtype   LayerNorm output feeding the next GEMM
//   qkvh    [T, 4D|F]   compute dtype   q|k|v (3D) + attention context (D); aliased by the FFN hidden
//   partial [S, H, C, C] fp32           split-K tied logits
//   probs   [H, C, ldp] compute dtype   softmax probabilities for the AV GEMM (16-bit paths only)
//   map     [H, C, C]   fp32            scratch attention map when the caller does not want it
//   cnt     [2 T / 256] int32           per (m-block, CTA rank) arrival counters of the fused residual + LayerNorm GEMM
//   split   fp32 path only              hi / lo halves of the current GEMM's activation and weight (tf32 x 3 product)
// ---------------------------------------------------------------------------------------------
static size_t tf32_scratch_bytes(long long M, int N, int K);

struct Plan {
  size_t el;  // bytes per element of the compute dtype
  int splits, ldp;
  int short_chunks;   // > 0: the tied row attention runs as ONE launch (row_attn_short.cu) with this many row chunks = splits
  size_t off_xn, off_qkvh, off_partial, off_probs, off_map, off_cnt, off_split, total;
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static inline bool is16(int dtype) { return dtype == RNAMSM_BF16 || dtype == RNAMSM_F16; }

static int pick_splits(int R, int C, int H, int dtype) {
  if (is16(dtype)) return row_logits_splits_16(R, C, H);
  const long long tiles = (long long)H * ceil_div(C, 128) * ceil_div(C, 128);
  int want = (int)std::max<long long>(1, (2 * 148) / std::max<long long>(1, tiles));
  want = std::max(1, std::min(want, std::max(1, R / 4)));
  const int rps = ceil_div(R, want);
  return ceil_div(R, rps);
}

static Plan make_plan(int R, int C, int D, int H, int F, int dtype, bool f32_tensor = false) {
  Plan p{};
  const size_t T = (size_t)R * C;
  p.el = is16(dtype) ? 2 : 4;
  p.short_chunks = is16(dtype) ? row_attn_short_chunks(R, C, H) : 0;
  p.splits = p.short_chunks > 0 ? p.short_chunks : pick_splits(R, C, H, dtype);
  p.ldp = is16(dtype) ? (C + 7) / 8 * 8 : C;
  size_t o = 0;
  p.off_xn = o;      o += align256(T * D * p.el);
  p.off_qkvh = o;    o += align256(T * (size_t)std::max(4 * D, F) * p.el);
  p.off_partial = o; o += align256((size_t)p.splits * H * C * C * 4);
  p.off_probs = o;   o += align256(is16(dtype) ? (size_t)H * C * p.ldp * p.el : 0);
  p.off_map = o;     o += align256((size_t)H * C * C * 4);
  p.off_cnt = o;     o += align256(ln_counter_bytes((long long)T));   // arrival counters of the fused LayerNorm epilogue
  p.off_split = o;   o += (dtype == RNAMSM_F32 && f32_tensor) ? tf32_scratch_bytes((long long)T, std::max(3 * D, F), std::max(D, F)) : 0;
  p.total = o;
  return p;
}

// fp32 path with RNAMSM_F32_TENSOR: the nn.Linear layers run on the tensor cores as a three-term tf32 product
// (umma_gemm.cu, kTf32) on hi / lo halves of both operands staged in the workspace's split region.
static size_t tf32_scratch_bytes(long long M, int N, int K) {
  return 2 * align256((size_t)M * K * 4) + 2 * align256((size_t)N * K * 4);
}
static int linear_tf32(const float* x, const float* W, long long M, int N, int K, const LinearEpilogue& e, float* out,
                       uint8_t* scratch, cudaStream_t st) {
  float* xh = reinterpret_cast<float*>(scratch);
  float* xl = reinterpret_cast<float*>(scratch + align256((size_t)M * K * 4));
  float* wh = reinterpret_cast<float*>(scratch + 2 * align256((size_t)M * K * 4));
  float* wl = reinterpret_cast<float*>(scratch + 2 * align256((size_t)M * K * 4) + align256((size_t)N * K * 4));
  int rc;
  if ((rc = launch_split_tf32(x, xh, xl, M * K, st))) return rc;
  if ((rc = launch_split_tf32(W, wh, wl, (long long)N * K, st))) return rc;
  return launch_linear_tf32(xh, xl, wh, wl, M, N, K, e, out, st);
}

static int linear_any(const void* x, const void* W, long long M, int N, int K, int dtype, const LinearEpilogue& e,
                      void* out, cudaStream_t st, const LnFuse* ln = nullptr, uint8_t* tf32_scratch = nullptr) {
  if (is16(dtype)) return launch_linear_16(x, W, M, N, K, dtype == RNAMSM_F16, e, out, st, ln);
  RNAMSM_REQUIRE(ln == nullptr, "linear: LayerNorm fusion exists in the 16-bit path only");
  if (dtype == RNAMSM_F32 && tf32_scratch != nullptr && N % 32 == 0 && K % 32 == 0)
    return linear_tf32((const float*)x, (const float*)W, M, N, K, e, (float*)out, tf32_scratch, st);
  if (dtype == RNAMSM_F32)
    return launch_linear_f32((const float*)x, (const float*)W, M, N, K, e, (float*)out, st);
  set_error("unknown dtype %d", dtype);
  return 2;
}

static int block_dtype(int requested, int dtype) {
  // per-block operand type: 0 (unset) inherits the layer dtype; the fp32 path is all-fp32
  if (dtype == RNAMSM_F32) return RNAMSM_F32;
  return is16(requested) ? requested : dtype;
}

// RNAMSM_FUSE_LN=1 routes every LayerNorm behind a residual GEMM through that GEMM's fused epilogue (umma_gemm.cu, kLN).
// OFF by default: the fused kernel is exact (bit-identical rows, tests/test_gpu_ops.py; bit-identical whole forwards,
// tests/test_gpu_forward_routes.py) but SLOWER on a B200 -- measured
// at 131072 x 768: residual GEMM 176 us + LayerNorm 94 us = 270 us un-fused vs 804 us fused (K = 768), 598 vs 935 us
// (K = 3072); the handshake itself is free (178 us with the row work skipped).  The 4 LayerNorm warps of a CTA keep only
// 8 rows (24 KiB) in flight while the GEMM's own TMA traffic holds HBM at 85 % of its peak, so each dependent
// load round trip takes ~5 us and the re-read runs at ~0.7 TB/s; hiding that latency needs ~90 KiB of rows in flight per
// SM (Little: 2.7 TB/s x 5 us / 148), which neither the register file nor the shared memory left beside the 6-stage
// operand ring can hold.  The stand-alone pass, with 64 warps per SM in flight, runs at 98 % of the HBM roofline.
static bool fuse_ln_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RNAMSM_FUSE_LN");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

// Debug range watch (rnamsm_debug_range_watch): when set, every 16-bit activation the layer writes (LayerNorm outputs,
// q|k|v, attention contexts, the post-GELU hidden) is scanned for values at the edge of its type's range.
static unsigned long long* g_range_counters = nullptr;
static int range_watch(const void* p, long long n, int dtype, cudaStream_t st) {
  if (g_range_counters == nullptr || !is16(dtype)) return 0;
  return launch_range_scan(p, n, dtype, g_range_counters, st);
}

// LayerNorm of the NEXT layer's row block, produced by this layer's fc2 epilogue (16-bit path)
struct NextLn { const float* w; const float* b; int dtype; };

// Column-attention probabilities a caller asked for (col_attn_probs.cu): P [H, C, R, R] and / or the column mean
// [H, R, R] (either NULL), lse: col_probs_scratch_bytes(R, C, H) bytes of scratch.
struct ColProbsOut { float* probs; float* mean; void* lse; };

// xn_ready: the workspace's xn region already holds LayerNorm_row(x) (written by the previous layer's fc2 epilogue).
static int layer_forward(const rnamsm_layer_weights* w, int D, int H, int F, float eps, float* x, int R, int C,
                         const uint8_t* pad, int dtype, float* row_probs_out, uint8_t* ws, const Plan& p,
                         cudaStream_t st, bool xn_ready = false, const NextLn* next = nullptr, bool f32_tensor = false,
                         const ColProbsOut* colp = nullptr) {
  const long long T = (long long)R * C;
  void* xn = ws + p.off_xn;
  uint8_t* qkv = ws + p.off_qkvh;
  void* ctx = qkv + (size_t)T * 3 * D * p.el;
  float* partial = reinterpret_cast<float*>(ws + p.off_partial);
  float* map = row_probs_out ? row_probs_out : reinterpret_cast<float*>(ws + p.off_map);
  const int row_dt = block_dtype(w->row.dtype, dtype);   // tied row attention: fp16 by default in the 16-bit path
  const int col_dt = block_dtype(w->col.dtype, dtype);
  void* probs_lp = is16(row_dt) ? (void*)(ws + p.off_probs) : nullptr;
  int rc;

  // With RNAMSM_FUSE_LN=1 every residual GEMM of the 16-bit path also emits the LayerNorm its successor needs
  // (umma_gemm.cu, kLN) and the stand-alone LayerNorm passes disappear except the very first one (see fuse_ln_enabled()
  // for why this is not the default).
  const bool fuse = is16(dtype) && fuse_ln_enabled();
  uint8_t* split = (dtype == RNAMSM_F32 && f32_tensor) ? ws + p.off_split : nullptr;   // operand halves of the tf32 x 3 product
  int* cnt = reinterpret_cast<int*>(ws + p.off_cnt);
  // the counters are zero between launches (the kernel resets them); a layer that starts a chain zeroes them once
  if (fuse && !xn_ready) RNAMSM_CHECK_CUDA(cudaMemsetAsync(cnt, 0, ln_counter_bytes(T), st));
  RNAMSM_REQUIRE(!xn_ready || fuse, "layer_forward: xn_ready needs the 16-bit path with LayerNorm fusion enabled");
  RNAMSM_REQUIRE(next == nullptr || fuse, "layer_forward: next-layer LayerNorm needs the 16-bit path with fusion enabled");

  // ---- tied row attention: x += out_proj(AV(softmax(sum_r q k^T)))   modules.py:385-401, 802-821
  if (!xn_ready && (rc = launch_layernorm(x, w->row.ln_w, w->row.ln_b, xn, row_dt, T, D, eps, st))) return rc;
  // align_scaling (modules.py:713-715) = 64^-1/2 / sqrt(R).  fp32 path: applied to q as the reference
  // does.  16-bit path: q carries the exact power of two 64^-1/2 and the 1/sqrt(R) factor is applied
  // to the fp32 logit sums in the softmax kernel (keeps q well inside the 16-bit normal range).
  const float q_scale = is16(row_dt) ? 0.125f : 0.125f / sqrtf((float)R);
  const float logit_scale = is16(row_dt) ? 1.0f / sqrtf((float)R) : 1.0f;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS, w->row.b_qkv, q_scale, D, pad};
    if ((rc = linear_any(xn, w->row.w_qkv, T, 3 * D, D, row_dt, e, qkv, st, nullptr, split))) return rc;
    if ((rc = range_watch(xn, T * D, row_dt, st)) || (rc = range_watch(qkv, T * 3 * D, row_dt, st))) return rc;
  }
  // key mask comes from MSA row 0 (padding_mask[:, 0], modules.py:780-784) = first C entries of pad
  if (is16(row_dt) && p.short_chunks > 0) {
    // short alignment (C <= 128): logits -> softmax -> A V in one cooperative launch (row_attn_short.cu)
    if ((rc = launch_row_attn_short_16(qkv, R, C, H, row_dt == RNAMSM_F16, partial, p.short_chunks, pad, logit_scale, map,
                                       probs_lp, p.ldp, ctx, st)))
      return rc;
  } else {
    if (is16(row_dt)) {
      if ((rc = launch_row_logits_16(qkv, R, C, H, row_dt == RNAMSM_F16, partial, p.splits, st))) return rc;
    } else {
      if ((rc = launch_row_logits_f32((const float*)qkv, R, C, H, partial, p.splits, st))) return rc;
    }
    if ((rc = launch_row_softmax(partial, p.splits, H, C, pad, logit_scale, map, probs_lp, p.ldp, row_dt, st))) return rc;
    if (is16(row_dt)) {
      if ((rc = launch_row_av_16(probs_lp, p.ldp, qkv, R, C, H, row_dt == RNAMSM_F16, ctx, st))) return rc;
    } else {
      if ((rc = launch_row_av_f32(map, C, (const float*)qkv, R, C, H, (float*)ctx, st))) return rc;
    }
  }
  // ---- column attention over the MSA depth                           modules.py:875-945
  // 16-bit path: LayerNorm writes its output in column-major token order (c * R + r), so the QKV GEMM
  // produces q|k|v as [C, R, 3D] and the flash kernel's K/V boxes read rows 3D elements apart instead of
  // C * 3D (one TMA row per 2 MiB page otherwise).  ctx comes back token-major for the out-projection.
  const int col_major = is16(col_dt) && R > 1 ? 1 : 0;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->row.b_out, 1.f, 0, nullptr};
    const LnFuse ln{w->col.ln_w, w->col.ln_b, eps, xn, col_dt == RNAMSM_F16, col_major ? R : 0, col_major ? C : 0, cnt};
    if ((rc = range_watch(ctx, T * D, row_dt, st))) return rc;
    if ((rc = linear_any(ctx, w->row.w_out, T, D, D, row_dt, e, x, st, fuse ? &ln : nullptr, split))) return rc;
  }
  if (!fuse &&
      (rc = launch_layernorm(x, w->col.ln_w, w->col.ln_b, xn, col_dt, T, D, eps, st, col_major ? R : 0, col_major ? C : 0)))
    return rc;
  if (R == 1) {
    // single-row shortcut: out_proj(v_proj(x)), modules.py:882-894.  Project with the v rows only.
    LinearEpilogue ev{RNAMSM_EPI_BIAS, w->col.b_qkv + 2 * D, 1.f, 0, nullptr};
    const void* wv = (const uint8_t*)w->col.w_qkv + (size_t)2 * D * D * p.el;
    if ((rc = linear_any(xn, wv, T, D, D, col_dt, ev, ctx, st, nullptr, split))) return rc;
  } else {
    LinearEpilogue e{RNAMSM_EPI_BIAS, w->col.b_qkv, 1.0f / sqrtf(64.f), D, nullptr};  // q *= scaling, :905
    if ((rc = linear_any(xn, w->col.w_qkv, T, 3 * D, D, col_dt, e, qkv, st, nullptr, split))) return rc;
    if (is16(col_dt)) {
      if ((rc = launch_col_attn_16(qkv, R, C, H, col_dt == RNAMSM_F16, col_major, pad, ctx, st))) return rc;
    } else {
      if ((rc = launch_col_attn_f32((const float*)qkv, R, C, H, pad, (float*)ctx, st))) return rc;
    }
  }
  // q|k of the column block are still in place (the flash kernel wrote ctx next to them)
  if (colp && (rc = launch_col_probs(qkv, R, C, H, col_dt, col_major, pad, colp->probs, colp->mean, colp->lse, st)))
    return rc;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->col.b_out, 1.f, 0, nullptr};
    const LnFuse ln{w->ffn_ln_w, w->ffn_ln_b, eps, xn, dtype == RNAMSM_F16, 0, 0, cnt};
    if ((rc = range_watch(xn, T * D, col_dt, st)) || (rc = range_watch(ctx, T * D, col_dt, st))) return rc;
    if (R > 1 && (rc = range_watch(qkv, T * 3 * D, col_dt, st))) return rc;
    if ((rc = linear_any(ctx, w->col.w_out, T, D, D, col_dt, e, x, st, fuse ? &ln : nullptr, split))) return rc;
  }

  // ---- feed-forward: x += fc2(gelu(fc1(LN(x))))                        modules.py:423-427
  if (!fuse && (rc = launch_layernorm(x, w->ffn_ln_w, w->ffn_ln_b, xn, dtype, T, D, eps, st))) return rc;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_GELU, w->fc1_b, 1.f, 0, nullptr};
    if ((rc = linear_any(xn, w->fc1_w, T, F, D, dtype, e, qkv, st, nullptr, split))) return rc;
    if ((rc = range_watch(xn, T * D, dtype, st)) || (rc = range_watch(qkv, T * (long long)F, dtype, st))) return rc;
  }
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->fc2_b, 1.f, 0, nullptr};
    LnFuse ln{nullptr, nullptr, eps, xn, 0, 0, 0, cnt};
    if (next) { ln.w = next->w; ln.b = next->b; ln.out_fp16 = next->dtype == RNAMSM_F16; }
    if ((rc = linear_any(qkv, w->fc2_w, T, D, F, dtype, e, x, st, next ? &ln : nullptr, split))) return rc;
  }
  return 0;
}


// ---------------------------------------------------------------------------------------------
// Several short MSAs in one pass (SURVEY.md 8f row 4).  The tokens of all MSAs sit back to back in one
// [T_total, D] stream: the token-local work (three LayerNorms, six GEMMs per layer) is launched ONCE over
// T_total, so a 256 x 51 alignment no longer pays a partial last wave and a pipeline ramp per GEMM; the
// attention steps, which are per alignment by definition (tied logits sum over that MSA's rows with its
// own 1/sqrt(R), modules.py:713-715; column attention runs over that MSA's depth), are launched per MSA on
// its slice.  Every output element is produced by exactly the instruction sequence of the one-MSA call, so
// the results are bit-identical to n_msa calls of rnamsm_msa_forward -- NOT the reference's padded [B,R,C]
// batch, whose align_scaling would use the padded row count.
// ---------------------------------------------------------------------------------------------
struct BatchPlan {
  size_t el;
  long long T;
  size_t off_xn, off_qkvh, off_partial, off_probs, off_map, off_pad, off_cnt, total;
  size_t partial_bytes, probs_bytes;
  std::vector<Plan> msa;      // every MSA's own plan, computed ONCE here and used by every layer
};

static int make_batch_plan(int n, const int* R, const int* C, int D, int H, int F, int dtype, BatchPlan* bp) {
  BatchPlan b{};
  b.el = 2;
  size_t partial = 0, probs = 0, map = 0;
  for (int i = 0; i < n; ++i) {
    if (R[i] < 2 || C[i] < 1) {
      set_error("msa_forward_batch: MSA %d has R=%d C=%d (need R >= 2, C >= 1; run single-row inputs through rnamsm_msa_forward)",
                i, R[i], C[i]);
      return 2;
    }
    const Plan p = make_plan(R[i], C[i], D, H, F, dtype);
    b.msa.push_back(p);
    partial = std::max(partial, align256((size_t)p.splits * H * C[i] * C[i] * 4));
    probs = std::max(probs, align256((size_t)H * C[i] * p.ldp * p.el));
    map = std::max(map, align256((size_t)H * C[i] * C[i] * 4));
    b.T += (long long)R[i] * C[i];
  }
  size_t o = 0;
  b.off_xn = o;      o += align256((size_t)b.T * D * b.el);
  b.off_qkvh = o;    o += align256((size_t)b.T * (size_t)std::max(4 * D, F) * b.el);
  b.off_partial = o; o += partial;
  b.off_probs = o;   o += probs;
  b.partial_bytes = partial; b.probs_bytes = probs;
  b.off_map = o;     o += map;
  b.off_pad = o;     o += align256((size_t)b.T);
  b.off_cnt = o;     o += align256(ln_counter_bytes(b.T));
  b.total = o;
  *bp = b;
  return 0;
}

static int layer_forward_batch(const rnamsm_layer_weights* w, int D, int H, int F, float eps, float* x, int n,
                               const int* R, const int* C, const uint8_t* has_pad, bool any_pad, int dtype, int layer,
                               float* const* row_attn_out, uint8_t* ws, const BatchPlan& bp,
                               cudaStream_t st, bool xn_ready = false, const NextLn* next = nullptr) {
  const long long T = bp.T;
  const size_t el = bp.el;
  uint8_t* xn = ws + bp.off_xn;
  uint8_t* qkv = ws + bp.off_qkvh;
  uint8_t* ctx = qkv + (size_t)T * 3 * D * el;
  float* partial = reinterpret_cast<float*>(ws + bp.off_partial);
  void* probs_lp = ws + bp.off_probs;
  const uint8_t* pad = ws + bp.off_pad;
  const int row_dt = block_dtype(w->row.dtype, dtype);
  const int col_dt = block_dtype(w->col.dtype, dtype);
  int rc;

  // token-local LayerNorms ride on the residual GEMMs as in layer_forward; the column block's LayerNorm stays a pass
  // per MSA because it transposes each MSA's own token order
  const bool fuse = fuse_ln_enabled();
  int* cnt = reinterpret_cast<int*>(ws + bp.off_cnt);
  if (fuse && !xn_ready) RNAMSM_CHECK_CUDA(cudaMemsetAsync(cnt, 0, ln_counter_bytes(T), st));
  // ---- tied row attention (same constants as layer_forward's 16-bit branch)
  if (!(xn_ready && fuse) && (rc = launch_layernorm(x, w->row.ln_w, w->row.ln_b, xn, row_dt, T, D, eps, st))) return rc;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS, w->row.b_qkv, 0.125f, D, any_pad ? pad : nullptr};
    if ((rc = linear_any(xn, w->row.w_qkv, T, 3 * D, D, row_dt, e, qkv, st))) return rc;
  }
  long long off = 0;
  for (int i = 0; i < n; ++i) {
    const Plan& p = bp.msa[i];
    RNAMSM_REQUIRE((size_t)p.splits * H * C[i] * C[i] * 4 <= bp.partial_bytes && (size_t)H * C[i] * p.ldp * el <= bp.probs_bytes,
                   "msa_forward_batch: MSA %d (splits %d) does not fit the planned partial / probs slabs", i, p.splits);
    const uint8_t* qkv_i = qkv + (size_t)off * 3 * D * el;
    const uint8_t* pad_i = (has_pad && has_pad[i]) ? pad + off : nullptr;
    float* map = (row_attn_out && row_attn_out[i])
                     ? row_attn_out[i] + (size_t)layer * H * C[i] * C[i]
                     : reinterpret_cast<float*>(ws + bp.off_map);
    if (p.short_chunks > 0) {   // the same one-launch kernel rnamsm_msa_forward uses for this shape (bit-identical results)
      if ((rc = launch_row_attn_short_16(qkv_i, R[i], C[i], H, row_dt == RNAMSM_F16, partial, p.short_chunks, pad_i,
                                         1.0f / sqrtf((float)R[i]), map, probs_lp, p.ldp, ctx + (size_t)off * D * el, st)))
        return rc;
    } else {
      if ((rc = launch_row_logits_16(qkv_i, R[i], C[i], H, row_dt == RNAMSM_F16, partial, p.splits, st))) return rc;
      if ((rc = launch_row_softmax(partial, p.splits, H, C[i], pad_i, 1.0f / sqrtf((float)R[i]), map, probs_lp, p.ldp,
                                   row_dt, st)))
        return rc;
      if ((rc = launch_row_av_16(probs_lp, p.ldp, qkv_i, R[i], C[i], H, row_dt == RNAMSM_F16, ctx + (size_t)off * D * el,
                                 st)))
        return rc;
    }
    off += (long long)R[i] * C[i];
  }
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->row.b_out, 1.f, 0, nullptr};
    if ((rc = linear_any(ctx, w->row.w_out, T, D, D, row_dt, e, x, st))) return rc;
  }

  // ---- column attention: LayerNorm per MSA (it transposes that MSA's token order), one QKV GEMM, flash
  // kernel per MSA on its [C, R, 3D] slice, one out-projection.
  off = 0;
  for (int i = 0; i < n; ++i) {
    const long long Ti = (long long)R[i] * C[i];
    if ((rc = launch_layernorm(x + (size_t)off * D, w->col.ln_w, w->col.ln_b, xn + (size_t)off * D * el, col_dt, Ti, D,
                               eps, st, R[i], C[i])))
      return rc;
    off += Ti;
  }
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS, w->col.b_qkv, 1.0f / sqrtf(64.f), D, nullptr};
    if ((rc = linear_any(xn, w->col.w_qkv, T, 3 * D, D, col_dt, e, qkv, st))) return rc;
  }
  off = 0;
  for (int i = 0; i < n; ++i) {
    const uint8_t* pad_i = (has_pad && has_pad[i]) ? pad + off : nullptr;
    if ((rc = launch_col_attn_16(qkv + (size_t)off * 3 * D * el, R[i], C[i], H, col_dt == RNAMSM_F16, 1, pad_i,
                                 ctx + (size_t)off * D * el, st)))
      return rc;
    off += (long long)R[i] * C[i];
  }
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->col.b_out, 1.f, 0, nullptr};
    const LnFuse ln{w->ffn_ln_w, w->ffn_ln_b, eps, xn, dtype == RNAMSM_F16, 0, 0, cnt};
    if ((rc = linear_any(ctx, w->col.w_out, T, D, D, col_dt, e, x, st, fuse ? &ln : nullptr))) return rc;
  }

  // ---- feed-forward over all tokens
  if (!fuse && (rc = launch_layernorm(x, w->ffn_ln_w, w->ffn_ln_b, xn, dtype, T, D, eps, st))) return rc;
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_GELU, w->fc1_b, 1.f, 0, nullptr};
    if ((rc = linear_any(xn, w->fc1_w, T, F, D, dtype, e, qkv, st))) return rc;
  }
  {
    LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, w->fc2_b, 1.f, 0, nullptr};
    LnFuse ln{nullptr, nullptr, eps, xn, 0, 0, 0, cnt};
    const bool emit = fuse && next != nullptr;
    if (emit) { ln.w = next->w; ln.b = next->b; ln.out_fp16 = next->dtype == RNAMSM_F16; }
    if ((rc = linear_any(qkv, w->fc2_w, T, D, F, dtype, e, x, st, emit ? &ln : nullptr))) return rc;
  }
  return 0;
}

// Embedding and layer stack of rnamsm_msa_forward_batch: everything but its final in-place LayerNorm.  Also the layer
// path of the scoring entry, which reads one token per grid and normalises only that row.
static int msa_forward_batch_layers(const rnamsm_model_weights* m, int n_msa, const int64_t* tokens, const int* R,
                                    const int* C, const uint8_t* has_pad, int dtype, float* x, float* const* row_attn_out,
                                    uint8_t* ws, const BatchPlan& bp, cudaStream_t st) {
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, N = m->num_layers;
  uint8_t* pad = ws + bp.off_pad;
  bool any_pad = false;
  long long off = 0;
  int rc;
  for (int i = 0; i < n_msa; ++i) {
    any_pad = any_pad || (has_pad && has_pad[i]);
    if ((rc = launch_embed_ln(tokens + off, R[i], C[i], m->tok_emb, m->vocab, m->pos_emb, m->n_pos, m->row_pos,
                              m->ln_before_w, m->ln_before_b, D, m->pad_idx, m->ln_eps, x + (size_t)off * D, pad + off, st)))
      return rc;
    off += (long long)R[i] * C[i];
  }
  for (int l = 0; l < N; ++l) {
    NextLn next{nullptr, nullptr, dtype};
    if (l + 1 < N)
      next = NextLn{m->layers[l + 1].row.ln_w, m->layers[l + 1].row.ln_b, block_dtype(m->layers[l + 1].row.dtype, dtype)};
    if ((rc = layer_forward_batch(&m->layers[l], D, H, F, m->ln_eps, x, n_msa, R, C, has_pad, any_pad, dtype, l,
                                  row_attn_out, ws, bp, st, l > 0, next.w ? &next : nullptr)))
      return rc;
  }
  return 0;
}

// RobertaLMHead (modules.py:313-319) on M rows: dense -> erf-GELU -> LayerNorm -> tied projection + bias.
// lm16: dense + GELU on tcgen05 from xn16 (the final LayerNorm's 16-bit output, 16-bit h), LayerNorm with fp32
// statistics -> fp32, 12-wide tied projection in fp32.  Otherwise FFMA (or tf32 x 3 with split scratch) from x, the
// final LayerNorm's fp32 output.  hbuf: M * D * 4 bytes, h32: M * D fp32.
static int lm_head_rows(const rnamsm_model_weights* m, const float* x, const void* xn16, long long M, int dtype, bool lm16,
                        uint8_t* hbuf, float* h32, uint8_t* tf32_split, float* logits_out, cudaStream_t st) {
  const int D = m->embed_dim;
  int rc;
  LinearEpilogue e{RNAMSM_EPI_BIAS_GELU, m->lm_dense_b, 1.f, 0, nullptr};
  if (lm16) {
    if ((rc = launch_linear_16(xn16, m->lm_dense_w16, M, D, D, dtype == RNAMSM_F16, e, hbuf, st))) return rc;
    if ((rc = launch_layernorm((const float*)hbuf, m->lm_ln_w, m->lm_ln_b, h32, RNAMSM_F32, M, D, m->ln_eps, st, 0, 0,
                               dtype)))
      return rc;
  } else {
    if ((rc = linear_any(x, m->lm_dense_w, M, D, D, RNAMSM_F32, e, hbuf, st, nullptr, tf32_split))) return rc;
    if ((rc = launch_layernorm((const float*)hbuf, m->lm_ln_w, m->lm_ln_b, h32, RNAMSM_F32, M, D, m->ln_eps, st))) return rc;
  }
  return launch_vocab_proj(h32, m->tok_emb, m->lm_bias, M, m->vocab, D, logits_out, st);
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

int rnamsm_version(void) { return RNAMSM_ABI_VERSION; }
const char* rnamsm_last_error(void) { return get_error(); }
long long rnamsm_launch_count(void) { return launch_count(); }
int rnamsm_gemm_pairs(void) { return gemm_max_pairs(); }

int rnamsm_profile_enable(int on) {
  for (auto& ev : g_prof_events) { g_prof_pool.push_back(ev.a); g_prof_pool.push_back(ev.b); }
  g_prof_events.clear();
  g_prof_on = on != 0;
  return 0;
}
int rnamsm_profile_num_classes(void) { return KC_COUNT; }
const char* rnamsm_profile_class_name(int i) { return (i >= 0 && i < KC_COUNT) ? kClassNames[i] : ""; }
int rnamsm_profile_collect(double* ms_out, long long* launches_out, int n) {
  RNAMSM_REQUIRE(n >= KC_COUNT, "profile_collect: need %d slots", (int)KC_COUNT);
  for (int i = 0; i < n; ++i) { ms_out[i] = 0.0; launches_out[i] = 0; }
  for (auto& ev : g_prof_events) {
    RNAMSM_CHECK_CUDA(cudaEventSynchronize(ev.b));
    float ms = 0.f;
    RNAMSM_CHECK_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
    ms_out[ev.cls] += ms;
    launches_out[ev.cls] += 1;
    g_prof_pool.push_back(ev.a);
    g_prof_pool.push_back(ev.b);
  }
  g_prof_events.clear();
  return 0;
}

int rnamsm_device_check(void) {
  int dev = 0;
  RNAMSM_CHECK_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0;
  RNAMSM_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  RNAMSM_CHECK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  RNAMSM_REQUIRE(major == 10, "rnamsm_b200 is built for sm_100a (B200); device %d is sm_%d%d", dev, major, minor);
  (void)gemm_max_pairs();   // resolve the CTA-pair occupancy now: every later plan and launch sees the same value
  return 0;
}

int rnamsm_embed_layernorm(const int64_t* tokens, int R, int C, const float* tok_emb, int vocab, const float* pos_emb,
                           int n_pos, const float* row_pos, const float* ln_w, const float* ln_b, int D, int pad_idx,
                           float eps, float* x_out, uint8_t* pad_out, void* stream) {
  return launch_embed_ln(tokens, R, C, tok_emb, vocab, pos_emb, n_pos, row_pos, ln_w, ln_b, D, pad_idx, eps, x_out,
                         pad_out, (cudaStream_t)stream);
}

int rnamsm_layernorm(const float* x, const float* w, const float* b, void* y, int y_dtype, long long n_rows, int D,
                     float eps, int tr_R, int tr_C, void* stream) {
  return launch_layernorm(x, w, b, y, y_dtype, n_rows, D, eps, (cudaStream_t)stream, tr_R, tr_C);
}

int rnamsm_linear(const void* x, const void* W, const float* bias, long long M, int N, int K, int dtype, int epilogue,
                  float q_scale, int q_cols, const uint8_t* row_mask, void* out, void* stream) {
  RNAMSM_REQUIRE(epilogue >= 0 && epilogue <= 2, "rnamsm_linear: unknown epilogue %d", epilogue);
  LinearEpilogue e{epilogue, bias, q_scale, q_cols, row_mask};
  return linear_any(x, W, M, N, K, dtype, e, out, (cudaStream_t)stream);
}

size_t rnamsm_linear_tf32_scratch_bytes(long long M, int N, int K) { return tf32_scratch_bytes(M, N, K); }

int rnamsm_linear_tf32(const float* x, const float* W, const float* bias, long long M, int N, int K, int epilogue,
                       float q_scale, int q_cols, const uint8_t* row_mask, float* out, void* scratch, size_t scratch_bytes,
                       void* stream) {
  RNAMSM_REQUIRE(epilogue >= 0 && epilogue <= 2, "linear_tf32: unknown epilogue %d", epilogue);
  RNAMSM_REQUIRE(scratch != nullptr && scratch_bytes >= tf32_scratch_bytes(M, N, K) &&
                     (reinterpret_cast<uintptr_t>(scratch) & 255) == 0,
                 "linear_tf32: scratch of %zu bytes (256 B aligned) required", tf32_scratch_bytes(M, N, K));
  LinearEpilogue e{epilogue, bias, q_scale, q_cols, row_mask};
  return linear_tf32(x, W, M, N, K, e, out, (uint8_t*)scratch, (cudaStream_t)stream);
}

int rnamsm_linear_residual_layernorm(const void* x, const void* W, const float* bias, long long M, int N, int K, int dtype,
                                     float* resid, const float* ln_w, const float* ln_b, float eps, void* y, int y_dtype,
                                     int tr_R, int tr_C, int* counters, void* stream) {
  RNAMSM_REQUIRE(is16(dtype) && is16(y_dtype), "linear_residual_layernorm: 16-bit operands and output only (dtype %d, y %d)",
                 dtype, y_dtype);
  LinearEpilogue e{RNAMSM_EPI_BIAS_RESIDUAL, bias, 1.f, 0, nullptr};
  const LnFuse ln{ln_w, ln_b, eps, y, y_dtype == RNAMSM_F16, tr_R, tr_C, counters};
  return launch_linear_16(x, W, M, N, K, dtype == RNAMSM_F16, e, resid, (cudaStream_t)stream, &ln);
}

int rnamsm_row_attn_splits(int R, int C, int H, int dtype) { return pick_splits(R, C, H, dtype); }

int rnamsm_row_attn_logits(const void* qkv, int R, int C, int H, int dtype, float* partial, int n_splits, void* stream) {
  if (is16(dtype)) return launch_row_logits_16(qkv, R, C, H, dtype == RNAMSM_F16, partial, n_splits, (cudaStream_t)stream);
  return launch_row_logits_f32((const float*)qkv, R, C, H, partial, n_splits, (cudaStream_t)stream);
}

int rnamsm_row_attn_short_chunks(int R, int C, int H) { return row_attn_short_chunks(R, C, H); }

int rnamsm_row_attn_short(const void* qkv, int R, int C, int H, int dtype, const uint8_t* key_pad, float logit_scale,
                          float* partial, int n_chunks, float* probs_out, void* probs_lp, int ld_lp, void* ctx,
                          void* stream) {
  RNAMSM_REQUIRE(is16(dtype), "rnamsm_row_attn_short: 16-bit dtypes only (the fp32 path keeps the three-kernel chain)");
  return launch_row_attn_short_16(qkv, R, C, H, dtype == RNAMSM_F16, partial, n_chunks, key_pad, logit_scale, probs_out,
                                  probs_lp, ld_lp, ctx, (cudaStream_t)stream);
}

int rnamsm_row_softmax(const float* partial, int n_splits, int H, int C, const uint8_t* key_pad, float logit_scale,
                       float* probs_out, void* probs_lp, int ld_lp, int dtype, void* stream) {
  return launch_row_softmax(partial, n_splits, H, C, key_pad, logit_scale, probs_out, probs_lp, ld_lp, dtype,
                            (cudaStream_t)stream);
}

int rnamsm_row_attn_av(const void* probs, int ldp, const void* qkv, int R, int C, int H, int dtype, void* ctx,
                       void* stream) {
  if (is16(dtype)) return launch_row_av_16(probs, ldp, qkv, R, C, H, dtype == RNAMSM_F16, ctx, (cudaStream_t)stream);
  return launch_row_av_f32((const float*)probs, ldp, (const float*)qkv, R, C, H, (float*)ctx, (cudaStream_t)stream);
}

int rnamsm_col_attn(const void* qkv, int R, int C, int H, int dtype, int qkv_col_major, const uint8_t* pad, void* ctx,
                    void* stream) {
  RNAMSM_REQUIRE(R >= 2, "rnamsm_col_attn: R=%d (the R == 1 shortcut is out_proj(v_proj(x)))", R);
  RNAMSM_REQUIRE(!qkv_col_major || is16(dtype), "rnamsm_col_attn: the column-major q|k|v layout exists in the 16-bit path only");
  if (is16(dtype))
    return launch_col_attn_16(qkv, R, C, H, dtype == RNAMSM_F16, qkv_col_major, pad, ctx, (cudaStream_t)stream);
  return launch_col_attn_f32((const float*)qkv, R, C, H, pad, (float*)ctx, (cudaStream_t)stream);
}

int rnamsm_col_attn_probs(const void* qkv, int R, int C, int H, int dtype, int qkv_col_major, const uint8_t* pad,
                          float* probs_out, float* mean_out, void* scratch, void* stream) {
  return launch_col_probs(qkv, R, C, H, dtype, qkv_col_major, pad, probs_out, mean_out, scratch, (cudaStream_t)stream);
}

int rnamsm_vocab_proj(const float* h, const float* E, const float* bias, long long M, int V, int D, float* out,
                      void* stream) {
  return launch_vocab_proj(h, E, bias, M, V, D, out, (cudaStream_t)stream);
}

size_t rnamsm_workspace_bytes(int R, int C, int D, int H, int F, int dtype) {
  if (R <= 0 || C <= 0) return 0;
  return make_plan(R, C, D, H, F, dtype & 0xff, (dtype & RNAMSM_F32_TENSOR) != 0).total;
}

size_t rnamsm_col_probs_scratch_bytes(int R, int C, int H) { return col_probs_scratch_bytes(R, C, H); }

int rnamsm_range_scan(const void* buf, long long n, int dtype, unsigned long long* counters, void* stream) {
  RNAMSM_REQUIRE(counters != nullptr, "range_scan: counters required");
  return launch_range_scan(buf, n, dtype, counters, (cudaStream_t)stream);
}
int rnamsm_debug_range_watch(unsigned long long* counters) {
  g_range_counters = counters;
  return 0;
}

int rnamsm_fused_layernorm(int dtype) { return (is16(dtype) && fuse_ln_enabled()) ? 1 : 0; }

}  // extern "C"

// col_probs_out / col_mean_out both NULL: exactly the launch sequence of rnamsm_layer_forward.  Otherwise the column
// probabilities' scratch sits right after the layer's own workspace.
static int layer_forward_entry(const rnamsm_layer_weights* w, int D, int H, int F, float ln_eps, float* x, int R, int C,
                               const uint8_t* pad, int dtype, float* row_probs_out, float* col_probs_out,
                               float* col_mean_out, void* workspace, size_t workspace_bytes, int xn_ready,
                               const float* next_ln_w, const float* next_ln_b, int next_ln_dtype, void* stream) {
  RNAMSM_REQUIRE(D == H * 64, "layer_forward: head_dim must be 64 (D=%d H=%d)", D, H);
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  dtype &= 0xff;
  RNAMSM_REQUIRE(dtype == RNAMSM_F32 || (is16(dtype) && !f32_tensor), "layer_forward: unknown dtype %d", dtype);
  const Plan p = make_plan(R, C, D, H, F, dtype, f32_tensor);
  const bool want_col = col_probs_out || col_mean_out;
  const size_t need = p.total + (want_col ? col_probs_scratch_bytes(R, C, H) : 0);
  RNAMSM_REQUIRE(workspace_bytes >= need, "layer_forward: workspace %zu < required %zu", workspace_bytes, need);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "layer_forward: workspace must be 256 B aligned");
  RNAMSM_REQUIRE((next_ln_w == nullptr) == (next_ln_b == nullptr), "layer_forward: next_ln_w and next_ln_b go together");
  const NextLn next{next_ln_w, next_ln_b, block_dtype(next_ln_dtype, dtype)};
  const ColProbsOut colp{col_probs_out, col_mean_out, (uint8_t*)workspace + p.total};
  return layer_forward(w, D, H, F, ln_eps, x, R, C, pad, dtype, row_probs_out, (uint8_t*)workspace, p,
                       (cudaStream_t)stream, xn_ready != 0, next_ln_w ? &next : nullptr, f32_tensor,
                       want_col ? &colp : nullptr);
}

static int msa_forward_entry(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                             float* x, float* row_attn_out, float* col_probs_out, float* col_mean_out,
                             float* const* rep_out, float* logits_out, void* workspace, size_t workspace_bytes,
                             void* stream, bool final_ln = true) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, N = m->num_layers;
  RNAMSM_REQUIRE(D == H * 64, "msa_forward: head_dim must be 64 (D=%d H=%d)", D, H);
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  dtype &= 0xff;
  RNAMSM_REQUIRE(dtype == RNAMSM_F32 || (is16(dtype) && !f32_tensor), "msa_forward: unknown dtype %d", dtype);
  RNAMSM_REQUIRE(R >= 1 && C >= 1, "msa_forward: empty MSA (R=%d C=%d)", R, C);
  const Plan p = make_plan(R, C, D, H, F, dtype, f32_tensor);
  const size_t T = (size_t)R * C;
  const size_t pad_bytes = (T + 255) & ~(size_t)255;
  const bool want_col = col_probs_out || col_mean_out;
  const size_t need = p.total + pad_bytes + (want_col ? col_probs_scratch_bytes(R, C, H) : 0);
  RNAMSM_REQUIRE(workspace_bytes >= need, "msa_forward: workspace %zu < required %zu", workspace_bytes, need);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "msa_forward: workspace must be 256 B aligned");
  uint8_t* ws = (uint8_t*)workspace;
  uint8_t* pad = ws + p.total;
  int rc;
  if ((rc = launch_embed_ln(tokens, R, C, m->tok_emb, m->vocab, m->pos_emb, m->n_pos, m->row_pos, m->ln_before_w,
                            m->ln_before_b, D, m->pad_idx, m->ln_eps, x, pad, st)))
    return rc;
  const uint8_t* pad_arg = has_pad ? pad : nullptr;
  for (int l = 0; l < N; ++l) {
    if (rep_out && rep_out[l]) RNAMSM_CHECK_CUDA(cudaMemcpyAsync(rep_out[l], x, T * D * 4, cudaMemcpyDeviceToDevice, st));
    float* map = row_attn_out ? row_attn_out + (size_t)l * H * C * C : nullptr;
    const ColProbsOut colp{col_probs_out ? col_probs_out + (size_t)l * H * C * R * R : nullptr,
                           col_mean_out ? col_mean_out + (size_t)l * H * R * R : nullptr, pad + pad_bytes};
    // layer l's fc2 epilogue also writes layer l+1's row-block LayerNorm (16-bit path)
    const bool fuse = is16(dtype) && fuse_ln_enabled();
    NextLn next{nullptr, nullptr, dtype};
    if (fuse && l + 1 < N)
      next = NextLn{m->layers[l + 1].row.ln_w, m->layers[l + 1].row.ln_b, block_dtype(m->layers[l + 1].row.dtype, dtype)};
    if ((rc = layer_forward(&m->layers[l], D, H, F, m->ln_eps, x, R, C, pad_arg, dtype, map, ws, p, st, fuse && l > 0,
                            next.w ? &next : nullptr, f32_tensor, want_col ? &colp : nullptr)))
      return rc;
  }
  if (!final_ln) return 0;   // the scoring entry normalises only the rows it reads (x stays pre-LayerNorm)
  // 16-bit path with logits wanted: the LM head's dense GEMM runs on the tensor cores, so it needs the final
  // LayerNorm's output in 16 bits as well -- written by a second (16-bit output) LayerNorm launch on the same rows
  // before the in-place fp32 one
  const bool lm16 = logits_out && is16(dtype) && m->lm_dense_w16 != nullptr;
  if (lm16 && (rc = launch_layernorm(x, m->ln_after_w, m->ln_after_b, ws + p.off_xn, dtype, (long long)T, D, m->ln_eps, st)))
    return rc;
  // emb_layer_norm_after in place (model.py:396): fp32 -> fp32, each warp reads its row before writing it
  if ((rc = launch_layernorm(x, m->ln_after_w, m->ln_after_b, x, RNAMSM_F32, (long long)T, D, m->ln_eps, st))) return rc;
  if (logits_out) {
    // LM head; scratch: the q|k|v|ctx region
    uint8_t* hbuf = ws + p.off_qkvh;
    float* h32 = reinterpret_cast<float*>(hbuf + align256(T * D * 4));
    if ((rc = lm_head_rows(m, x, ws + p.off_xn, (long long)T, dtype, lm16, hbuf, h32,
                           (dtype == RNAMSM_F32 && f32_tensor) ? ws + p.off_split : nullptr, logits_out, st)))
      return rc;
  }
  return 0;
}

extern "C" {

int rnamsm_layer_forward(const rnamsm_layer_weights* w, int D, int H, int F, float ln_eps, float* x, int R, int C,
                         const uint8_t* pad, int dtype, float* row_probs_out, void* workspace, size_t workspace_bytes,
                         int xn_ready, const float* next_ln_w, const float* next_ln_b, int next_ln_dtype, void* stream) {
  return layer_forward_entry(w, D, H, F, ln_eps, x, R, C, pad, dtype, row_probs_out, nullptr, nullptr, workspace,
                             workspace_bytes, xn_ready, next_ln_w, next_ln_b, next_ln_dtype, stream);
}

int rnamsm_layer_forward_col_probs(const rnamsm_layer_weights* w, int D, int H, int F, float ln_eps, float* x, int R, int C,
                                   const uint8_t* pad, int dtype, float* row_probs_out, float* col_probs_out,
                                   float* col_mean_out, void* workspace, size_t workspace_bytes, int xn_ready,
                                   const float* next_ln_w, const float* next_ln_b, int next_ln_dtype, void* stream) {
  return layer_forward_entry(w, D, H, F, ln_eps, x, R, C, pad, dtype, row_probs_out, col_probs_out, col_mean_out,
                             workspace, workspace_bytes, xn_ready, next_ln_w, next_ln_b, next_ln_dtype, stream);
}

int rnamsm_msa_forward(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                       float* x, float* row_attn_out, float* const* rep_out, float* logits_out, void* workspace,
                       size_t workspace_bytes, void* stream) {
  return msa_forward_entry(m, tokens, R, C, has_pad, dtype, x, row_attn_out, nullptr, nullptr, rep_out, logits_out,
                           workspace, workspace_bytes, stream);
}

int rnamsm_msa_forward_col_probs(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                 int dtype, float* x, float* row_attn_out, float* col_probs_out, float* col_mean_out,
                                 float* const* rep_out, float* logits_out, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  return msa_forward_entry(m, tokens, R, C, has_pad, dtype, x, row_attn_out, col_probs_out, col_mean_out, rep_out,
                           logits_out, workspace, workspace_bytes, stream);
}

size_t rnamsm_batch_workspace_bytes(int n_msa, const int* R, const int* C, int D, int H, int F, int dtype) {
  BatchPlan bp;
  if (n_msa <= 0 || !is16(dtype) || make_batch_plan(n_msa, R, C, D, H, F, dtype, &bp)) return 0;
  return bp.total;
}

int rnamsm_msa_forward_batch(const rnamsm_model_weights* m, int n_msa, const int64_t* tokens, const int* R, const int* C,
                             const uint8_t* has_pad, int dtype, float* x, float* const* row_attn_out, void* workspace,
                             size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim;
  RNAMSM_REQUIRE(D == H * 64, "msa_forward_batch: head_dim must be 64 (D=%d H=%d)", D, H);
  RNAMSM_REQUIRE(is16(dtype), "msa_forward_batch: 16-bit operand types only (dtype %d); the fp32 parity path runs one MSA per call",
                 dtype);
  RNAMSM_REQUIRE(n_msa >= 1 && R && C, "msa_forward_batch: empty batch");
  BatchPlan bp;
  int rc;
  if ((rc = make_batch_plan(n_msa, R, C, D, H, F, dtype, &bp))) return rc;
  RNAMSM_REQUIRE(workspace_bytes >= bp.total, "msa_forward_batch: workspace %zu < required %zu", workspace_bytes, bp.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "msa_forward_batch: workspace must be 256 B aligned");
  if ((rc = msa_forward_batch_layers(m, n_msa, tokens, R, C, has_pad, dtype, x, row_attn_out, (uint8_t*)workspace, bp, st)))
    return rc;
  return launch_layernorm(x, m->ln_after_w, m->ln_after_b, x, RNAMSM_F32, bp.T, D, m->ln_eps, st);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// LM-head scoring of one alignment (rnamsm_msa_masked_marginals).  Entry k is the LM-head output at (row, cols[k]) of
// the grid with that token masked (or of the grid itself, mask_idx < 0).  The entry runs ceil(n_cols / group) passes;
// a pass builds its variant grids on the device, runs them through the layer stack, gathers the one pre-final-LayerNorm
// row each grid is scored at, and runs the final LayerNorm and the LM head on those rows only.
//   16-bit, R >= 2: the pass's grids go through the batch layer path together (token-local kernels once per pass,
//                   attention per grid), exactly as rnamsm_msa_forward_batch runs them.
//   fp32 / tf32 x 3, or R == 1: one forward per grid (msa_forward_entry without its final LayerNorm and head).
// Every kernel a row meets is row-local or has fixed tiles independent of the row count, so the logits are bit-identical
// to rnamsm_msa_forward's logits of the masked grid at that token.
// Workspace for `group` grids of R x C tokens (every region 256 B aligned):
//   tok   [g, T] int64           the pass's variant grids
//   x     [g or 1, T, D] fp32    hidden states: the pass's g grids (batch route) or the current grid
//   fwd                          the forward's own workspace: the batch plan of g grids, or the one-MSA plan + pad flags
//   rows  [g, D] fp32            the gathered rows (normalised in place when the head runs in fp32)
//   xn16  [g, D] 16-bit          the final LayerNorm's 16-bit output (16-bit dtypes)
//   h     [g, D] <= 4 B          LM-head dense + GELU
//   h32   [g, D] fp32            LM-head LayerNorm
//   split                        tf32 x 3 operand halves of the dense GEMM (RNAMSM_F32_TENSOR)
// The logits land in the caller's logprobs_out and become log-probabilities in place.
// ---------------------------------------------------------------------------------------------
namespace rnamsm {

// The layer route of the LM-head entries (scoring, sampling, the categorical Jacobian): n grids of R x C tokens, back to
// back in tok, through the embedding and the layer stack without the final LayerNorm; x [n, T, D] receives their
// pre-final-LayerNorm hidden states.  maps (optional): grid i's row-attention maps [N, H, C, C] at maps + i * N H C C.
//   batch (16-bit, R >= 2): the n grids together through the batch layer path; fwd holds its plan for n grids.
//   otherwise: one msa_forward_entry per grid; fwd holds the one-MSA plan + pad flags (fwd_bytes).
static int grids_forward_layers(const rnamsm_model_weights* m, const int64_t* tok, int n, int R, int C, int has_pad,
                                int dtype, bool batch, float* x, uint8_t* fwd, size_t fwd_bytes, cudaStream_t st,
                                float* maps = nullptr) {
  const int D = m->embed_dim;
  const size_t T = (size_t)R * C;
  const size_t map_sz = (size_t)m->num_layers * m->num_heads * C * C;
  int rc;
  if (!batch) {
    for (int i = 0; i < n; ++i)
      if ((rc = msa_forward_entry(m, tok + i * T, R, C, has_pad, dtype, x + i * T * D, maps ? maps + i * map_sz : nullptr,
                                  nullptr, nullptr, nullptr, nullptr, fwd, fwd_bytes, st, false)))
        return rc;
    return 0;
  }
  const int dt = dtype & 0xff;
  std::vector<int> Rs(n, R), Cs(n, C);
  std::vector<uint8_t> pads(n, has_pad ? 1 : 0);
  std::vector<float*> map_ptrs;
  if (maps)
    for (int i = 0; i < n; ++i) map_ptrs.push_back(maps + i * map_sz);
  BatchPlan bp;
  if ((rc = make_batch_plan(n, Rs.data(), Cs.data(), D, m->num_heads, m->ffn_dim, dt, &bp))) return rc;
  return msa_forward_batch_layers(m, n, tok, Rs.data(), Cs.data(), pads.data(), dt, x, maps ? map_ptrs.data() : nullptr,
                                  fwd, bp, st);
}

struct ScorePlan {
  bool batch;
  size_t fwd_bytes, off_tok, off_x, off_fwd, off_rows, off_xn16, off_h, off_h32, off_split, total;
};

static int make_score_plan(int R, int C, int D, int H, int F, int dtype, int group, ScorePlan* out) {
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const int dt = dtype & 0xff;
  RNAMSM_REQUIRE((dtype & ~(0xff | RNAMSM_F32_TENSOR)) == 0 && (dt == RNAMSM_F32 || (is16(dt) && !f32_tensor)),
                 "score: unknown dtype %d", dtype);
  RNAMSM_REQUIRE(R >= 1 && C >= 1 && D > 0 && H > 0 && F > 0 && group >= 1, "score: bad shape R=%d C=%d D=%d H=%d F=%d group=%d",
                 R, C, D, H, F, group);
  const size_t T = (size_t)R * C, g = (size_t)group;
  ScorePlan s{};
  s.batch = is16(dt) && R >= 2;
  if (s.batch) {
    std::vector<int> Rs(group, R), Cs(group, C);
    BatchPlan bp;
    int rc;
    if ((rc = make_batch_plan(group, Rs.data(), Cs.data(), D, H, F, dt, &bp))) return rc;
    s.fwd_bytes = bp.total;
  } else {
    s.fwd_bytes = make_plan(R, C, D, H, F, dt, f32_tensor).total + align256(T);
  }
  size_t o = 0;
  s.off_tok = o;   o += align256(g * T * 8);
  s.off_x = o;     o += align256((s.batch ? g : 1) * T * D * 4);
  s.off_fwd = o;   o += align256(s.fwd_bytes);
  s.off_rows = o;  o += align256(g * D * 4);
  s.off_xn16 = o;  o += is16(dt) ? align256(g * D * 2) : 0;
  s.off_h = o;     o += align256(g * D * 4);
  s.off_h32 = o;   o += align256(g * D * 4);
  s.off_split = o; o += (dt == RNAMSM_F32 && f32_tensor) ? tf32_scratch_bytes((long long)g, D, D) : 0;
  s.total = o;
  *out = s;
  return 0;
}

}  // namespace rnamsm

extern "C" {

size_t rnamsm_score_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group) {
  ScorePlan sp;
  if (make_score_plan(R, C, D, H, F, dtype, group, &sp)) return 0;
  return sp.total;
}

int rnamsm_msa_masked_marginals(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                int dtype, int row, const int* cols, int n_cols, int mask_idx, int group,
                                float* logits_out, float* logprobs_out, void* workspace, size_t workspace_bytes,
                                void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, V = m->vocab;
  RNAMSM_REQUIRE(D == H * 64, "masked_marginals: head_dim must be 64 (D=%d H=%d)", D, H);
  ScorePlan sp;
  int rc;
  if ((rc = make_score_plan(R, C, D, H, F, dtype, group, &sp))) return rc;
  RNAMSM_REQUIRE(row >= 0 && row < R, "masked_marginals: row %d outside the %d MSA rows", row, R);
  RNAMSM_REQUIRE(n_cols >= 0 && (n_cols == 0 || (cols && logprobs_out)), "masked_marginals: cols and logprobs_out required");
  RNAMSM_REQUIRE(workspace_bytes >= sp.total, "masked_marginals: workspace %zu < required %zu", workspace_bytes, sp.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "masked_marginals: workspace must be 256 B aligned");
  if (n_cols == 0) return 0;
  const int dt = dtype & 0xff;
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const long long T = (long long)R * C;
  uint8_t* ws = (uint8_t*)workspace;
  int64_t* grids = reinterpret_cast<int64_t*>(ws + sp.off_tok);
  float* x = reinterpret_cast<float*>(ws + sp.off_x);
  float* rows = reinterpret_cast<float*>(ws + sp.off_rows);
  void* xn16 = ws + sp.off_xn16;
  const bool lm16 = is16(dt) && m->lm_dense_w16 != nullptr;   // the head msa_forward_entry runs for this dtype
  // x holds one grid on the per-grid route, so that route runs the grids of a pass one call at a time
  auto layers = [&](const int64_t* tok, int n) -> int {
    return grids_forward_layers(m, tok, n, R, C, has_pad, dtype, sp.batch, x, ws + sp.off_fwd, sp.fwd_bytes, st);
  };
  if (mask_idx < 0 && (rc = layers(tokens, 1))) return rc;   // wt-marginals: one forward, every column read from it
  for (int k0 = 0; k0 < n_cols; k0 += group) {
    const int n = std::min(group, n_cols - k0);
    const int* ck = cols + k0;
    if (mask_idx < 0) {
      if ((rc = launch_score_gather(x, 0, row, C, ck, n, D, rows, st))) return rc;
    } else {
      if ((rc = launch_score_variants(tokens, T, row, C, ck, nullptr, n, mask_idx, m->pad_idx, grids, st))) return rc;
      if (sp.batch) {
        if ((rc = layers(grids, n))) return rc;
        if ((rc = launch_score_gather(x, T, row, C, ck, n, D, rows, st))) return rc;
      } else {
        for (int i = 0; i < n; ++i) {
          if ((rc = layers(grids + (size_t)i * T, 1))) return rc;
          if ((rc = launch_score_gather(x, 0, row, C, ck + i, 1, D, rows + (size_t)i * D, st))) return rc;
        }
      }
    }
    // final LayerNorm on the n rows (the 16-bit operand of the tensor-core head, or fp32 in place), LM head, log_softmax
    if ((rc = launch_layernorm(rows, m->ln_after_w, m->ln_after_b, lm16 ? xn16 : (void*)rows, lm16 ? dt : RNAMSM_F32, n, D,
                               m->ln_eps, st)))
      return rc;
    float* lp = logprobs_out + (size_t)k0 * V;
    if ((rc = lm_head_rows(m, rows, xn16, n, dt, lm16, ws + sp.off_h, reinterpret_cast<float*>(ws + sp.off_h32),
                           (dt == RNAMSM_F32 && f32_tensor) ? ws + sp.off_split : nullptr, lp, st)))
      return rc;
    if ((rc = launch_score_log_softmax(lp, logits_out ? logits_out + (size_t)k0 * V : nullptr, n, V, tokens, row, C, ck,
                                       m->pad_idx, st)))
      return rc;
  }
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Iterative masked sampling of one alignment with the LM head (rnamsm_msa_gibbs_sample; the algorithm and its random
// numbers are in sample.cu).  Chains run `group` at a time; a pass loops over all steps of its chains, enqueuing only.
// One step of a pass of g chains:
//   copy the g states into the grid buffer, mask kernel -> the g masked grids
//   layer stack: 16-bit with R >= 2, the g grids through the batch layer path together; fp32 / tf32 x 3 or R == 1, one
//   msa_forward_entry per grid without its final LayerNorm (the routes of the scoring entry)
//   row gather (only when n_rows < R) -> the sampled rows' pre-final-LayerNorm states
//   final LayerNorm and LM head on those g * n_rows * C rows only, draw kernel -> the g states
// Workspace for `group` grids of R x C tokens, M = group * n_rows * C head rows (every region 256 B aligned):
//   tok   [g, T] int64           the pass's masked grids
//   x     [g, T, D] fp32         hidden states of the pass's grids
//   fwd                          the forward's own workspace: the batch plan of g grids, or the one-MSA plan + pad flags
//   hx    [M, D] fp32            the gathered rows (n_rows < R only; otherwise the head reads x)
//   xn16  [M, D] 16-bit          the final LayerNorm's 16-bit output (16-bit dtypes)
//   h     [M, D] <= 4 B          LM-head dense + GELU, then the logits [M, V]
//   h32   [M, D] fp32            LM-head LayerNorm
//   split                        tf32 x 3 operand halves of the dense GEMM (RNAMSM_F32_TENSOR)
// ---------------------------------------------------------------------------------------------
namespace rnamsm {

struct SamplePlan {
  bool batch;
  size_t fwd_bytes, off_tok, off_x, off_fwd, off_hx, off_xn16, off_h, off_h32, off_split, total;
};

static int make_sample_plan(int R, int C, int D, int H, int F, int dtype, int group, int n_rows, SamplePlan* out) {
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const int dt = dtype & 0xff;
  RNAMSM_REQUIRE((dtype & ~(0xff | RNAMSM_F32_TENSOR)) == 0 && (dt == RNAMSM_F32 || (is16(dt) && !f32_tensor)),
                 "sample: unknown dtype %d", dtype);
  RNAMSM_REQUIRE(R >= 1 && C >= 1 && D > 0 && H > 0 && F > 0 && group >= 1 && n_rows >= 1 && n_rows <= R,
                 "sample: bad shape R=%d C=%d D=%d H=%d F=%d group=%d n_rows=%d", R, C, D, H, F, group, n_rows);
  const size_t T = (size_t)R * C, g = (size_t)group, M = g * n_rows * C;
  SamplePlan s{};
  s.batch = is16(dt) && R >= 2;
  if (s.batch) {
    std::vector<int> Rs(group, R), Cs(group, C);
    BatchPlan bp;
    int rc;
    if ((rc = make_batch_plan(group, Rs.data(), Cs.data(), D, H, F, dt, &bp))) return rc;
    s.fwd_bytes = bp.total;
  } else {
    s.fwd_bytes = make_plan(R, C, D, H, F, dt, f32_tensor).total + align256(T);
  }
  size_t o = 0;
  s.off_tok = o;   o += align256(g * T * 8);
  s.off_x = o;     o += align256(g * T * D * 4);
  s.off_fwd = o;   o += align256(s.fwd_bytes);
  s.off_hx = o;    o += n_rows < R ? align256(M * D * 4) : 0;
  s.off_xn16 = o;  o += is16(dt) ? align256(M * D * 2) : 0;
  s.off_h = o;     o += align256(M * D * 4);
  s.off_h32 = o;   o += align256(M * D * 4);
  s.off_split = o; o += (dt == RNAMSM_F32 && f32_tensor) ? tf32_scratch_bytes((long long)M, D, D) : 0;
  s.total = o;
  *out = s;
  return 0;
}

}  // namespace rnamsm

extern "C" {

size_t rnamsm_sample_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group, int n_rows) {
  SamplePlan sp;
  if (make_sample_plan(R, C, D, H, F, dtype, group, n_rows, &sp)) return 0;
  return sp.total;
}

int rnamsm_msa_gibbs_sample(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                            const int* rows, int n_rows, int n_chains, int steps, int start_step, float mask_prob,
                            float temperature, unsigned allowed_bitmask, unsigned long long seed, int group,
                            int64_t* tokens_out, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, V = m->vocab;
  const int mask_idx = V - 1;   // the RNA alphabet appends <mask> after its residues (msm/data.py)
  RNAMSM_REQUIRE(D == H * 64, "gibbs_sample: head_dim must be 64 (D=%d H=%d)", D, H);
  SamplePlan sp;
  int rc;
  if ((rc = make_sample_plan(R, C, D, H, F, dtype, group, n_rows, &sp))) return rc;
  RNAMSM_REQUIRE(rows && tokens_out, "gibbs_sample: rows and tokens_out required");
  RNAMSM_REQUIRE(n_chains >= 1 && steps >= 0 && start_step >= 0 && steps <= INT_MAX - start_step,
                 "gibbs_sample: n_chains=%d steps=%d start_step=%d", n_chains, steps, start_step);
  RNAMSM_REQUIRE(mask_prob >= 0.f && mask_prob <= 1.f, "gibbs_sample: mask_prob %g outside [0, 1]", (double)mask_prob);
  RNAMSM_REQUIRE(temperature >= 0.f, "gibbs_sample: temperature %g < 0", (double)temperature);
  RNAMSM_REQUIRE(V >= 2 && V <= 32 && V <= D, "gibbs_sample: vocabulary of %d tokens (2 .. 32, <= D)", V);
  RNAMSM_REQUIRE(allowed_bitmask != 0 && (V == 32 || (allowed_bitmask >> V) == 0) &&
                     !((allowed_bitmask >> m->pad_idx) & 1u) && !((allowed_bitmask >> mask_idx) & 1u),
                 "gibbs_sample: allowed_bitmask 0x%x must be a non-empty set of vocabulary tokens other than <pad> and <mask>",
                 allowed_bitmask);
  RNAMSM_REQUIRE(workspace_bytes >= sp.total, "gibbs_sample: workspace %zu < required %zu", workspace_bytes, sp.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "gibbs_sample: workspace must be 256 B aligned");
  const int dt = dtype & 0xff;
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const long long T = (long long)R * C;
  if (tokens)
    for (int k = 0; k < n_chains; ++k)
      RNAMSM_CHECK_CUDA(cudaMemcpyAsync(tokens_out + (size_t)k * T, tokens, (size_t)T * 8, cudaMemcpyDeviceToDevice, st));
  uint8_t* ws = (uint8_t*)workspace;
  int64_t* grids = reinterpret_cast<int64_t*>(ws + sp.off_tok);
  float* x = reinterpret_cast<float*>(ws + sp.off_x);
  float* hx = n_rows < R ? reinterpret_cast<float*>(ws + sp.off_hx) : x;
  void* xn16 = ws + sp.off_xn16;
  uint8_t* h = ws + sp.off_h;
  const bool lm16 = is16(dt) && m->lm_dense_w16 != nullptr;   // the head msa_forward_entry runs for this dtype
  for (int k0 = 0; k0 < n_chains; k0 += group) {
    const int n = std::min(group, n_chains - k0);
    const long long M = (long long)n * n_rows * C;
    for (int s = start_step; s < start_step + steps; ++s) {
      RNAMSM_CHECK_CUDA(cudaMemcpyAsync(grids, tokens_out + (size_t)k0 * T, (size_t)n * T * 8, cudaMemcpyDeviceToDevice, st));
      if ((rc = launch_sample_mask(tokens_out, grids, n, R, C, rows, n_rows, m->pad_idx, mask_idx, mask_prob, seed, k0, s, st)))
        return rc;
      if ((rc = grids_forward_layers(m, grids, n, R, C, has_pad, dtype, sp.batch, x, ws + sp.off_fwd, sp.fwd_bytes, st)))
        return rc;
      if (n_rows < R && (rc = launch_sample_gather_rows(x, n, R, C, rows, n_rows, D, hx, st))) return rc;
      // final LayerNorm on the M head rows (the 16-bit operand of the tensor-core head, or fp32 in place), LM head, draw
      if ((rc = launch_layernorm(hx, m->ln_after_w, m->ln_after_b, lm16 ? xn16 : (void*)hx, lm16 ? dt : RNAMSM_F32, M, D,
                                 m->ln_eps, st)))
        return rc;
      float* logits = reinterpret_cast<float*>(h);   // h is free again once the head's LayerNorm has read it
      if ((rc = lm_head_rows(m, hx, xn16, M, dt, lm16, h, reinterpret_cast<float*>(ws + sp.off_h32),
                             (dt == RNAMSM_F32 && f32_tensor) ? ws + sp.off_split : nullptr, logits, st)))
        return rc;
      if ((rc = launch_sample_draw(logits, V, temperature, allowed_bitmask, tokens_out, n, R, C, rows, n_rows, m->pad_idx,
                                   mask_prob, seed, k0, s, st)))
        return rc;
    }
  }
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Categorical Jacobian of the LM head for one query row (rnamsm_msa_categorical_jacobian; the definition and the
// contact map are in jacobian.cu).  Entry e names slab s = i * A + a of J: the grid with token (row, positions[i])
// replaced by alphabet[a].  J is zeroed first, so every slab no entry names (the wild type's) is exactly 0.  One forward
// of `tokens` gives the wild-type logits of the query row; the entries then run `group` grids per pass:
//   variant kernel (score.cu, with per-entry tokens) -> the pass's substituted grids
//   layer stack on the route of the scoring and sampling entries (grids_forward_layers)
//   row gather (R >= 2 only) -> the query row of each grid, M = g * C head rows
//   final LayerNorm and LM head on those rows, collect kernel -> f - f_wt into the entries' slabs
// Workspace: the sampling plan of `group` grids with one sampled row (tok / x / fwd / hx / xn16 / h / h32 / split for
// M = g * C head rows; the pass's logits [M, V] land in h), then
//   wt    [C, V <= D] fp32               the wild-type logits of the query row (sized [C, D])
//   list  int32 [1 + P + A + 3 n]        row | positions | alphabet | per entry: column, token, slab
// ---------------------------------------------------------------------------------------------
namespace rnamsm {

struct JacobianPlan {
  SamplePlan sp;
  size_t off_wt, off_list, total;
};

static int make_jacobian_plan(int R, int C, int D, int H, int F, int dtype, int group, int P, int A, int n_entries,
                              JacobianPlan* out) {
  RNAMSM_REQUIRE(P >= 1 && A >= 1 && n_entries >= 0, "jacobian: P=%d A=%d n_entries=%d", P, A, n_entries);
  JacobianPlan j{};
  int rc;
  if ((rc = make_sample_plan(R, C, D, H, F, dtype, group, 1, &j.sp))) return rc;
  size_t o = j.sp.total;
  j.off_wt = o;   o += align256((size_t)C * D * 4);
  j.off_list = o; o += align256((1 + (size_t)P + A + 3 * (size_t)n_entries) * 4);
  j.total = o;
  *out = j;
  return 0;
}

}  // namespace rnamsm

extern "C" {

size_t rnamsm_jacobian_workspace_bytes(int R, int C, int D, int H, int F, int dtype, int group, int P, int A,
                                       int n_entries) {
  JacobianPlan jp;
  if (make_jacobian_plan(R, C, D, H, F, dtype, group, P, A, n_entries, &jp)) return 0;
  return jp.total;
}

int rnamsm_msa_categorical_jacobian(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad,
                                    int dtype, int row, const int* positions, int P, const int* alphabet, int A,
                                    const int* entries, int n_entries, int group, float* jacobian_out, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, V = m->vocab;
  RNAMSM_REQUIRE(D == H * 64, "categorical_jacobian: head_dim must be 64 (D=%d H=%d)", D, H);
  JacobianPlan jp;
  int rc;
  if ((rc = make_jacobian_plan(R, C, D, H, F, dtype, group, P, A, n_entries, &jp))) return rc;
  RNAMSM_REQUIRE(V >= 1 && V <= D, "categorical_jacobian: vocabulary of %d tokens (<= D=%d)", V, D);
  RNAMSM_REQUIRE(row >= 0 && row < R, "categorical_jacobian: row %d outside the %d MSA rows", row, R);
  RNAMSM_REQUIRE(tokens && positions && alphabet && jacobian_out && (n_entries == 0 || entries),
                 "categorical_jacobian: tokens, positions, alphabet, entries and jacobian_out required");
  RNAMSM_REQUIRE(workspace_bytes >= jp.total, "categorical_jacobian: workspace %zu < required %zu", workspace_bytes, jp.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "categorical_jacobian: workspace must be 256 B aligned");
  // the host list, checked here and staged into the workspace with one copy
  std::vector<int> list(1 + (size_t)P + A + 3 * (size_t)n_entries);
  int* l_pos = list.data() + 1;
  int* l_alph = l_pos + P;
  int* l_col = l_alph + A;
  int* l_tok = l_col + n_entries;
  int* l_slab = l_tok + n_entries;
  list[0] = row;
  for (int i = 0; i < P; ++i) {
    RNAMSM_REQUIRE(positions[i] >= 0 && positions[i] < C, "categorical_jacobian: position %d outside the %d columns",
                   positions[i], C);
    l_pos[i] = positions[i];
  }
  for (int a = 0; a < A; ++a) {
    RNAMSM_REQUIRE(alphabet[a] >= 0 && alphabet[a] < V, "categorical_jacobian: token %d outside the vocabulary of %d",
                   alphabet[a], V);
    l_alph[a] = alphabet[a];
  }
  for (int e = 0; e < n_entries; ++e) {
    const int s = entries[e];
    RNAMSM_REQUIRE(s >= 0 && s < P * A && (e == 0 || s > entries[e - 1]),
                   "categorical_jacobian: entry %d (slab %d) must be ascending in [0, P*A = %d)", e, s, P * A);
    l_col[e] = positions[s / A];
    l_tok[e] = alphabet[s % A];
    l_slab[e] = s;
  }
  const int dt = dtype & 0xff;
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const long long T = (long long)R * C;
  const SamplePlan& sp = jp.sp;
  uint8_t* ws = (uint8_t*)workspace;
  int64_t* grids = reinterpret_cast<int64_t*>(ws + sp.off_tok);
  float* x = reinterpret_cast<float*>(ws + sp.off_x);
  float* hx = R > 1 ? reinterpret_cast<float*>(ws + sp.off_hx) : x;
  void* xn16 = ws + sp.off_xn16;
  uint8_t* h = ws + sp.off_h;
  float* wt = reinterpret_cast<float*>(ws + jp.off_wt);
  int* d_list = reinterpret_cast<int*>(ws + jp.off_list);
  const int* d_pos = d_list + 1;
  const int* d_alph = d_pos + P;
  const int* d_col = d_alph + A;
  const int* d_tok = d_col + n_entries;
  const int* d_slab = d_tok + n_entries;
  const bool lm16 = is16(dt) && m->lm_dense_w16 != nullptr;   // the head msa_forward_entry runs for this dtype
  RNAMSM_CHECK_CUDA(cudaMemcpyAsync(d_list, list.data(), list.size() * 4, cudaMemcpyHostToDevice, st));
  RNAMSM_CHECK_CUDA(cudaMemsetAsync(jacobian_out, 0, (size_t)P * A * P * A * 4, st));
  if (n_entries == 0) return 0;
  // the query row of the n grids in x -> final LayerNorm (the 16-bit operand of the tensor-core head, or fp32 in place)
  // -> LM head -> logits [n * C, V]
  auto head = [&](int n, float* logits) -> int {
    const long long M = (long long)n * C;
    int r;
    if (R > 1 && (r = launch_sample_gather_rows(x, n, R, C, d_list, 1, D, hx, st))) return r;
    if ((r = launch_layernorm(hx, m->ln_after_w, m->ln_after_b, lm16 ? xn16 : (void*)hx, lm16 ? dt : RNAMSM_F32, M, D,
                              m->ln_eps, st)))
      return r;
    return lm_head_rows(m, hx, xn16, M, dt, lm16, h, reinterpret_cast<float*>(ws + sp.off_h32),
                        (dt == RNAMSM_F32 && f32_tensor) ? ws + sp.off_split : nullptr, logits, st);
  };
  if ((rc = grids_forward_layers(m, tokens, 1, R, C, has_pad, dtype, sp.batch, x, ws + sp.off_fwd, sp.fwd_bytes, st)))
    return rc;
  if ((rc = head(1, wt))) return rc;
  float* logits = reinterpret_cast<float*>(h);   // h is free again once the head's LayerNorm has read it
  for (int k0 = 0; k0 < n_entries; k0 += group) {
    const int n = std::min(group, n_entries - k0);
    if ((rc = launch_score_variants(tokens, T, row, C, d_col + k0, d_tok + k0, n, 0, m->pad_idx, grids, st))) return rc;
    if ((rc = grids_forward_layers(m, grids, n, R, C, has_pad, dtype, sp.batch, x, ws + sp.off_fwd, sp.fwd_bytes, st)))
      return rc;
    if ((rc = head(n, logits))) return rc;
    if ((rc = launch_jacobian_collect(logits, wt, n, C, V, d_pos, P, d_alph, A, d_slab + k0, jacobian_out, st))) return rc;
  }
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Full-length features of an alignment longer than the learned column positions, from overlapping windows
// (rnamsm_msa_forward_windows; the window plan and the definition and arithmetic of the stitched outputs are in
// windows.cu).  The K windows run `group` at a time; a pass of g windows:
//   build kernel -> the pass's window grids [g, R, W + 1]
//   layer stack on the route of the LM-head entries (grids_forward_layers), with each grid's maps
//   row gather (R >= 2 only) -> row 0 of each grid; final LayerNorm on those g (W + 1) rows only
//   contact head per window (contacts wanted)
//   stitch kernel -> emb_out, atp_out (and contacts_out)
// Every step is the one rnamsm_msa_forward runs on that grid, so each window's outputs are bit-identical to a forward of
// its grid.  Workspace for `group` (at most K) windows, every region 256 B aligned:
//   tok   [g, R, W + 1] int64        the pass's window grids
//   x     [g, R, W + 1, D] fp32      their pre-final-LayerNorm hidden states
//   fwd                              the forward's own workspace: the batch plan of g grids, or the one-MSA plan + pads
//   maps  [g, N H, W + 1, W + 1]     their row-attention maps, BOS row and column included
//   hx    [g, W + 1, D] fp32         row 0 of each grid, normalised in place (R >= 2; otherwise x itself)
//   cw    [g, W, W] fp32             each window's contacts (contacts wanted)
//   ca    [N H (W + 1)] fp32         the contact head's scratch (contacts wanted)
//   list  int32 [K + 1]              the window starts, then 0 (the row the gather reads)
// ---------------------------------------------------------------------------------------------
namespace rnamsm {

struct WindowPlan {
  bool batch;
  int W, K, group;
  size_t fwd_bytes, off_tok, off_x, off_fwd, off_maps, off_hx, off_cw, off_ca, off_list, total;
};

static int make_window_plan(int R, int C, int D, int H, int F, int N, int dtype, int group, int window, int stride,
                            bool want_contacts, WindowPlan* out) {
  const bool f32_tensor = (dtype & RNAMSM_F32_TENSOR) != 0;
  const int dt = dtype & 0xff;
  RNAMSM_REQUIRE((dtype & ~(0xff | RNAMSM_F32_TENSOR)) == 0 && (dt == RNAMSM_F32 || (is16(dt) && !f32_tensor)),
                 "windows: unknown dtype %d", dtype);
  RNAMSM_REQUIRE(R >= 1 && C >= 2 && D > 0 && H > 0 && F > 0 && N > 0 && group >= 1,
                 "windows: bad shape R=%d C=%d D=%d H=%d F=%d N=%d group=%d", R, C, D, H, F, N, group);
  WindowPlan w{};
  w.K = window_starts(C - 1, window, stride, nullptr);
  if (w.K == 0) return 2;
  w.W = std::min(window, C - 1);
  w.group = std::min(group, w.K);
  const int Cw = w.W + 1;
  const size_t T = (size_t)R * Cw, g = (size_t)w.group, NH = (size_t)N * H;
  w.batch = is16(dt) && R >= 2;
  if (w.batch) {
    std::vector<int> Rs(w.group, R), Cs(w.group, Cw);
    BatchPlan bp;
    int rc;
    if ((rc = make_batch_plan(w.group, Rs.data(), Cs.data(), D, H, F, dt, &bp))) return rc;
    w.fwd_bytes = bp.total;
  } else {
    w.fwd_bytes = make_plan(R, Cw, D, H, F, dt, f32_tensor).total + align256(T);
  }
  size_t o = 0;
  w.off_tok = o;  o += align256(g * T * 8);
  w.off_x = o;    o += align256(g * T * D * 4);
  w.off_fwd = o;  o += align256(w.fwd_bytes);
  w.off_maps = o; o += align256(g * NH * Cw * Cw * 4);
  w.off_hx = o;   o += R > 1 ? align256(g * Cw * D * 4) : 0;
  w.off_cw = o;   o += want_contacts ? align256(g * w.W * w.W * 4) : 0;
  w.off_ca = o;   o += want_contacts ? align256(NH * Cw * 4) : 0;
  w.off_list = o; o += align256(((size_t)w.K + 1) * 4);
  w.total = o;
  *out = w;
  return 0;
}

}  // namespace rnamsm

extern "C" {

size_t rnamsm_windows_workspace_bytes(int R, int C, int D, int H, int F, int N, int dtype, int group, int window, int stride,
                                      int want_contacts) {
  WindowPlan wp;
  if (make_window_plan(R, C, D, H, F, N, dtype, group, window, stride, want_contacts != 0, &wp)) return 0;
  return wp.total;
}

int rnamsm_msa_forward_windows(const rnamsm_model_weights* m, const int64_t* tokens, int R, int C, int has_pad, int dtype,
                               int window, int stride, int group, float* emb_out, float* atp_out, float* contacts_out,
                               const float* contact_w, const float* contact_b, void* workspace, size_t workspace_bytes,
                               void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int D = m->embed_dim, H = m->num_heads, F = m->ffn_dim, N = m->num_layers, NH = N * H;
  RNAMSM_REQUIRE(D == H * 64, "forward_windows: head_dim must be 64 (D=%d H=%d)", D, H);
  const int max_window = m->n_pos - m->pad_idx - 2;   // positions of a [R, W + 1] grid run up to W + 1 + pad_idx
  RNAMSM_REQUIRE(window >= 1 && window <= max_window, "forward_windows: window %d outside [1, %d] (the learned positions)",
                 window, max_window);
  WindowPlan wp;
  int rc;
  if ((rc = make_window_plan(R, C, D, H, F, N, dtype, group, window, stride, contacts_out != nullptr, &wp))) return rc;
  RNAMSM_REQUIRE(tokens && emb_out && atp_out, "forward_windows: tokens, emb_out and atp_out required");
  RNAMSM_REQUIRE(!contacts_out || contact_w, "forward_windows: contacts need the regression weights contact_w");
  RNAMSM_REQUIRE(workspace_bytes >= wp.total, "forward_windows: workspace %zu < required %zu", workspace_bytes, wp.total);
  RNAMSM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "forward_windows: workspace must be 256 B aligned");
  const int L = C - 1, W = wp.W, K = wp.K, Cw = W + 1;
  std::vector<int> list((size_t)K + 1);
  window_starts(L, window, stride, list.data());
  list[K] = 0;
  uint8_t* ws = (uint8_t*)workspace;
  int64_t* grids = reinterpret_cast<int64_t*>(ws + wp.off_tok);
  float* x = reinterpret_cast<float*>(ws + wp.off_x);
  float* maps = reinterpret_cast<float*>(ws + wp.off_maps);
  float* hx = R > 1 ? reinterpret_cast<float*>(ws + wp.off_hx) : x;
  float* cw = contacts_out ? reinterpret_cast<float*>(ws + wp.off_cw) : nullptr;
  float* ca = reinterpret_cast<float*>(ws + wp.off_ca);
  int* d_starts = reinterpret_cast<int*>(ws + wp.off_list);
  RNAMSM_CHECK_CUDA(cudaMemcpyAsync(d_starts, list.data(), list.size() * 4, cudaMemcpyHostToDevice, st));
  for (int k0 = 0; k0 < K; k0 += wp.group) {
    const int n = std::min(wp.group, K - k0);
    if ((rc = launch_window_build(tokens, R, C, d_starts, k0, n, W, grids, st))) return rc;
    if ((rc = grids_forward_layers(m, grids, n, R, Cw, has_pad, dtype, wp.batch, x, ws + wp.off_fwd, wp.fwd_bytes, st, maps)))
      return rc;
    if (R > 1 && (rc = launch_sample_gather_rows(x, n, R, Cw, d_starts + K, 1, D, hx, st))) return rc;
    if ((rc = launch_layernorm(hx, m->ln_after_w, m->ln_after_b, hx, RNAMSM_F32, (long long)n * Cw, D, m->ln_eps, st)))
      return rc;
    for (int i = 0; contacts_out && i < n; ++i)
      if ((rc = rnamsm_contact_head(maps + (size_t)i * NH * Cw * Cw, NH, Cw, 1, W, contact_w, contact_b,
                                    cw + (size_t)i * W * W, ca, st)))
        return rc;
    if ((rc = launch_window_stitch(maps, NH, cw, hx, D, d_starts, K, k0, n, W, L, emb_out, atp_out, contacts_out, st)))
      return rc;
  }
  return 0;
}

}  // extern "C"
