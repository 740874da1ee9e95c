// MSA ingest on the device (SURVEY.md 8f "next" row 1): the step immediately in front of the hot path.
// HBM-bound byte / integer work, one warp per MSA row, no tensor cores:
//   msa_clean_kernel      MSA.from_fasta's per-character rules (utils/align.py:311-313): drop lowercase, '.',
//                         '*'; T -> U; RYKMSWBDHVN -> X -- a per-row stream compaction with warp ballots
//   greedy select         MSA.greedy_select (utils/align.py:128-148), the "diversity-max/min" sub-sampler:
//                         num-1 rounds of { mismatch count of every row against the last pick (uint16, kept for
//                         all rounds), mean over the picks, arg-max / arg-min with first index on ties }.  Exact
//                         ties between candidates are common (duplicate rows), and in the reference they are
//                         decided by float64 rounding: np.delete(...) hands .mean(0) a Fortran-ordered array, so
//                         numpy sums along the picks with its 8-accumulator pairwise scheme.  np_pairwise_sum
//                         reproduces that scheme operation for operation, so the selection is index-identical
//   msa_tokenize_kernel   gather the selected rows, 256-entry LUT (Vocab.encode, utils/tokenization.py:107-129),
//                         prepend <cls>: int64 [R, L+1], the exact input tensor of rnamsm_msa_forward
#include "../../include/rnamsm_b200.h"
#include "common.cuh"
#include "launch.h"

namespace rnamsm {

// Bio.SeqIO's FASTA parser (what MSA.from_fasta iterates) reads the file in text mode, so '\r\n' and a lone '\r' end a
// line like '\n'.  It rstrip()s every line, joins them and removes ' ' and '\r' (SimpleFastaParser).  So a space and a
// line end are always dropped, while the other blanks str.isspace() knows ('\t', '\v', '\f', 0x1c-0x1f) are dropped
// only where nothing but blanks follows them up to the end of their line: a tab inside a line is kept.
__device__ __forceinline__ bool is_soft_blank(uint8_t c) { return c == '\t' || c == '\v' || c == '\f' || (c >= 0x1c && c <= 0x1f); }
__device__ __forceinline__ bool is_line_end(uint8_t c) { return c == '\n' || c == '\r'; }

// append the soft blanks of raw[from, to) (all blanks, spaces among them) to the row: a run whose line went on
__device__ int append_blank_run(const uint8_t* __restrict__ raw, long long from, long long to, uint8_t* __restrict__ row,
                                int L, int written, int lane) {
  for (long long p = from; p < to; p += 32) {
    const long long q = p + lane;
    const uint8_t ch = q < to ? raw[q] : (uint8_t)' ';
    const bool keep = ch != ' ';
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    const int pos = written + __popc(m & ((1u << lane) - 1u));
    if (keep && pos < L) row[pos] = ch;
    written += __popc(m);
  }
  return written;
}

// raw: concatenated record bodies; off[n] .. off[n+1]: bytes of record n.  out [N, L]; bad[0] != 0 if a
// cleaned row is not exactly L long.
__global__ void __launch_bounds__(256)
msa_clean_kernel(const uint8_t* __restrict__ raw, const long long* __restrict__ off, int N, int L,
                 uint8_t* __restrict__ out, int* __restrict__ bad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + warp;
  if (n >= N) return;
  const long long b = off[n], e = off[n + 1];
  uint8_t* row = out + (size_t)n * L;
  int written = 0;
  long long run = -1;          // start of a trailing blank run of earlier steps, kept only if text follows it
  for (long long p = b; p < e; p += 32) {
    const long long q = p + lane;
    uint8_t ch = q < e ? raw[q] : (uint8_t)'\n';             // the body ends where its last line ends
    const bool soft = is_soft_blank(ch), solid = !soft && ch != ' ';
    const unsigned solid_m = __ballot_sync(0xffffffffu, solid);
    const unsigned text_m = __ballot_sync(0xffffffffu, solid && !is_line_end(ch));
    if (run >= 0 && solid_m) {                               // the first solid byte decides the pending run
      if ((text_m >> (__ffs(solid_m) - 1)) & 1u) written = append_blank_run(raw, run, p, row, L, written, lane);
      run = -1;
    }
    // a soft blank is kept if the next solid byte of this step is text; none: the run stays pending
    const unsigned later = lane == 31 ? 0u : solid_m & (0xffffffffu << (lane + 1));
    const bool soft_kept = soft && later && ((text_m >> (__ffs(later) - 1)) & 1u);
    if (solid_m == 0u) {
      if (run < 0) run = p;
    } else if (solid_m >> 31 == 0u) {
      run = p + 32 - __clz(solid_m);
    }
    // then MSA.from_fasta's own rules: drop lowercase, '.', '*'; T -> U; IUPAC -> X
    const bool keep = soft_kept || (solid && !is_line_end(ch) && !((ch >= 'a' && ch <= 'z') || ch == '.' || ch == '*'));
    if (ch == 'T') ch = 'U';
    else if (ch == 'R' || ch == 'Y' || ch == 'K' || ch == 'M' || ch == 'S' || ch == 'W' || ch == 'B' || ch == 'D' ||
             ch == 'H' || ch == 'V' || ch == 'N') ch = 'X';
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    const int pos = written + __popc(m & ((1u << lane) - 1u));
    if (keep && pos < L) row[pos] = ch;
    written += __popc(m);
  }
  if (lane == 0 && written != L) atomicExch(bad, n + 1);
}

struct Best { double v; int i; };

__device__ __forceinline__ Best better(Best a, Best b, bool want_max) {
  // larger (max) / smaller (min) value wins; equal values: the smaller index (np.argmax / argmin: first occurrence)
  if (b.i < 0) return a;
  if (a.i < 0) return b;
  if (want_max ? (b.v > a.v) : (b.v < a.v)) return b;
  if (b.v == a.v && b.i < a.i) return b;
  return a;
}

// round k, phase 1 (one warp per row): dist[k-1][n] = number of mismatches between row n and the last pick
__global__ void __launch_bounds__(256)
greedy_hamming_kernel(const uint8_t* __restrict__ chars, int N, int L, const int* __restrict__ selected, int k,
                      uint16_t* __restrict__ dist) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint8_t* ref = chars + (size_t)selected[k - 1] * L;
  uint16_t* out = dist + (size_t)(k - 1) * N;
  for (int n = blockIdx.x * 8 + warp; n < N; n += gridDim.x * 8) {
    const uint8_t* row = chars + (size_t)n * L;
    int mism = 0;
    for (int l = lane; l < L; l += 32) mism += row[l] != ref[l];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mism += __shfl_xor_sync(0xffffffffu, mism, o);
    if (lane == 0) out[n] = (uint16_t)mism;
  }
}

// numpy's pairwise float64 sum of a[0..n) = lut[col[i * stride]] (loops_utils.h.src: < 8 sequential; <= 128: eight
// running accumulators over blocks of 8, tree-combined, then the tail; larger: split at a multiple of 8 and recurse)
__device__ double np_pairwise_sum(const uint16_t* col, size_t stride, int n, const double* __restrict__ lut) {
  if (n < 8) {
    double res = 0.0;
    for (int i = 0; i < n; ++i) res += lut[col[i * stride]];
    return res;
  }
  if (n <= 128) {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = lut[col[j * stride]];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] += lut[col[(size_t)(i + j) * stride]];
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += lut[col[(size_t)i * stride]];
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  return np_pairwise_sum(col, stride, n2, lut) + np_pairwise_sum(col + (size_t)n2 * stride, stride, n - n2, lut);
}

// round k, phase 2 (one thread per row): value = mean_j dist[j][n] / L over the k picks, exactly as the reference's
// np.delete(pairwise_distances, indices, axis=1).mean(0) evaluates it (Fortran-ordered -> pairwise sum along k)
__global__ void __launch_bounds__(256)
greedy_mean_kernel(const uint16_t* __restrict__ dist, int N, int L, int k, const uint8_t* __restrict__ is_sel,
                   int want_max, Best* __restrict__ block_best) {
  extern __shared__ double lut[];            // lut[m] = (double)m / (double)L   == cdist(..., "hamming")
  __shared__ Best sb[8];
  for (int m = threadIdx.x; m <= L; m += blockDim.x) lut[m] = (double)m / (double)L;
  __syncthreads();
  Best mine{0.0, -1};
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    if (is_sel[n]) continue;
    const double mean = np_pairwise_sum(dist + n, (size_t)N, k, lut) / (double)k;
    mine = better(mine, Best{mean, n}, want_max != 0);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best other;
    other.v = __shfl_xor_sync(0xffffffffu, mine.v, o);
    other.i = __shfl_xor_sync(0xffffffffu, mine.i, o);
    mine = better(mine, other, want_max != 0);
  }
  if (lane == 0) sb[warp] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    Best b = sb[0];
    for (int w = 1; w < 8; ++w) b = better(b, sb[w], want_max != 0);
    block_best[blockIdx.x] = b;
  }
}

__global__ void __launch_bounds__(32)
greedy_pick_kernel(const Best* __restrict__ block_best, int n_blocks, int* __restrict__ selected, int k,
                   uint8_t* __restrict__ is_sel, int want_max) {
  const int lane = threadIdx.x;
  Best b{0.0, -1};
  for (int i = lane; i < n_blocks; i += 32) b = better(b, block_best[i], want_max != 0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best other;
    other.v = __shfl_xor_sync(0xffffffffu, b.v, o);
    other.i = __shfl_xor_sync(0xffffffffu, b.i, o);
    b = better(b, other, want_max != 0);
  }
  if (lane == 0) {
    selected[k] = b.i;
    is_sel[b.i] = 1;
  }
}

// sort <= 1024 picks ascending (indices = sorted(indices), utils/align.py:146): one block, odd-even transposition
__global__ void __launch_bounds__(1024)
sort_small_kernel(int* __restrict__ v, int n) {
  __shared__ int s[1024];
  const int t = threadIdx.x;
  s[t] = t < n ? v[t] : 0x7fffffff;
  __syncthreads();
  for (int phase = 0; phase < n; ++phase) {
    const int i = 2 * t + (phase & 1);
    if (i + 1 < n && s[i] > s[i + 1]) { const int x = s[i]; s[i] = s[i + 1]; s[i + 1] = x; }
    __syncthreads();
  }
  if (t < n) v[t] = s[t];
}

// tokens[r, 0] = bos; tokens[r, 1 + l] = lut[chars[rows[r], l]]   (rows == nullptr: identity)
__global__ void __launch_bounds__(256)
msa_tokenize_kernel(const uint8_t* __restrict__ chars, int L, const int* __restrict__ rows, int R,
                    const uint8_t* __restrict__ lut, int bos, int64_t* __restrict__ tokens) {
  __shared__ uint8_t slut[256];
  slut[threadIdx.x] = lut[threadIdx.x];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + warp;
  if (r >= R) return;
  const uint8_t* src = chars + (size_t)(rows ? rows[r] : r) * L;
  int64_t* dst = tokens + (size_t)r * (L + 1);
  if (lane == 0) dst[0] = bos;
  for (int l = lane; l < L; l += 32) dst[1 + l] = slut[src[l]];
}

}  // namespace rnamsm

using namespace rnamsm;

extern "C" {

int rnamsm_msa_clean(const uint8_t* raw, const long long* offsets, int N, int L, uint8_t* chars_out, int* bad_row,
                     void* stream) {
  RNAMSM_REQUIRE(N > 0 && L > 0, "msa_clean: empty MSA (N=%d L=%d)", N, L);
  cudaStream_t st = (cudaStream_t)stream;
  RNAMSM_CHECK_CUDA(cudaMemsetAsync(bad_row, 0, sizeof(int), st));
  msa_clean_kernel<<<ceil_div(N, 8), 256, 0, st>>>(raw, offsets, N, L, chars_out, bad_row);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

size_t rnamsm_msa_greedy_workspace(int N, int num) {
  size_t o = ((size_t)N + 255) & ~(size_t)255;                       // is_sel
  o += (size_t)(148 * 4) * sizeof(Best) + 256;                        // per-block candidates
  o += (size_t)(num > 1 ? num - 1 : 1) * (size_t)N * sizeof(uint16_t);   // mismatch counts of every round
  return o;
}

int rnamsm_msa_greedy_select(const uint8_t* chars, int N, int L, int num, int want_max, int* selected_out,
                             void* workspace, void* stream) {
  RNAMSM_REQUIRE(N > 0 && L > 0 && num >= 1 && num <= 1024, "msa_greedy_select: N=%d L=%d num=%d (num <= 1024)", N, L, num);
  RNAMSM_REQUIRE(num <= N, "msa_greedy_select: num=%d > depth %d (take the MSA as it is)", num, N);
  RNAMSM_REQUIRE(L < 65536 && (size_t)(L + 1) * sizeof(double) <= 200 * 1024, "msa_greedy_select: L=%d too long", L);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  uint8_t* is_sel = ws;
  size_t o = ((size_t)N + 255) & ~(size_t)255;
  Best* block_best = reinterpret_cast<Best*>(ws + o);
  o += (size_t)(148 * 4) * sizeof(Best) + 256;
  o &= ~(size_t)255;
  uint16_t* dist = reinterpret_cast<uint16_t*>(ws + o);
  const int blocks_h = std::min(ceil_div(N, 8), 148 * 4);
  const int blocks_m = std::min(ceil_div(N, 256), 148 * 4);
  const size_t lut_bytes = (size_t)(L + 1) * sizeof(double);
  // the LUT shares the 48 KiB default with greedy_mean_kernel's static sb[8]: 6128 <= L <= 6143 needs the opt-in too
  if (lut_bytes + 8 * sizeof(Best) > 48 * 1024)
    RNAMSM_CHECK_CUDA(cudaFuncSetAttribute(greedy_mean_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lut_bytes));
  RNAMSM_CHECK_CUDA(cudaMemsetAsync(is_sel, 0, (size_t)N, st));
  const int zero = 0;
  RNAMSM_CHECK_CUDA(cudaMemcpyAsync(selected_out, &zero, sizeof(int), cudaMemcpyHostToDevice, st));   // indices = [0]
  const uint8_t one = 1;
  RNAMSM_CHECK_CUDA(cudaMemcpyAsync(is_sel, &one, 1, cudaMemcpyHostToDevice, st));
  for (int k = 1; k < num; ++k) {
    greedy_hamming_kernel<<<blocks_h, 256, 0, st>>>(chars, N, L, selected_out, k, dist);
    greedy_mean_kernel<<<blocks_m, 256, lut_bytes, st>>>(dist, N, L, k, is_sel, want_max, block_best);
    greedy_pick_kernel<<<1, 32, 0, st>>>(block_best, blocks_m, selected_out, k, is_sel, want_max);
  }
  sort_small_kernel<<<1, 1024, 0, st>>>(selected_out, num);
  count_launch(3 * (num - 1) + 1);
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int rnamsm_msa_tokenize(const uint8_t* chars, int L, const int* rows, int R, const uint8_t* lut256, int bos,
                        int64_t* tokens_out, void* stream) {
  RNAMSM_REQUIRE(R > 0 && L > 0, "msa_tokenize: empty selection");
  msa_tokenize_kernel<<<ceil_div(R, 8), 256, 0, (cudaStream_t)stream>>>(chars, L, rows, R, lut256, bos, tokens_out);
  count_launch();
  RNAMSM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
