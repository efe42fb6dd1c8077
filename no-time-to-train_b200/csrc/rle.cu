// COCO run-length encoding of the output masks straight from the packed full-resolution words
// (SURVEY.md §8f rank 1).
//
// Reference: `_output_inqueue` copies `binary_masks [K_out,H,W] bool` to the host (105 MB per image) and
// `encode_results` calls pycocotools `mask_utils.encode(np.asfortranarray(mask))` per mask
// (no_time_to_train/pl_wrapper/sam2matcher_pl.py:144-158, no_time_to_train/dataset/coco_ref_dataset.py:590-613).
// The wire format is pycocotools' (pinned 2.0.8, pyproject.toml:35; source not under /root/reference):
//   rleEncode   — runs over the mask in COLUMN-major order, alternating zeros/ones, starting with zeros
//                 (first count 0 if pixel (0,0) is set); the reference's own `mask_to_rle_pytorch`
//                 (sam2/utils/amg.py:111-140) produces the same counts and pins this half;
//   rleToString — per count x = cnts[i] - (i > 2 ? cnts[i-2] : 0), emitted LEB128-like in 5-bit groups, low group
//                 first: c = x & 0x1f; x >>= 5; more = (c & 0x10) ? x != -1 : x != 0; if (more) c |= 0x20; c += 48.
//
// One CTA per output mask.  Only the mask's rect can hold ones, so only its columns (plus one column and one
// row of zeros that close the last runs) are visited.  A warp takes a 32-column strip and walks down the rect in
// 32-row blocks: each lane loads the packed word of one row, a 5-step shuffle butterfly transposes the 32x32 bit
// block so that each lane holds 32 rows of ONE column, and `col ^ (col << 1 | carry)` marks the run boundaries.
// Pass 1 counts boundaries per column, a block scan turns the counts into output offsets, pass 2 writes the
// boundary positions x*H + y in column-major order; differences of neighbours are the counts.  The string stage
// sizes every count, scans the sizes and writes the characters.
#include "common.cuh"

namespace nttt {

constexpr int kRleThreads = 256;
constexpr int kRleWarps = kRleThreads / 32;

// lane r holds row r of a 32x32 bit block (bit c = column c); returns, in lane c, column c (bit r = row r)
__device__ __forceinline__ uint32_t transpose32(uint32_t w, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const uint32_t low = s == 16 ? 0x0000ffffu : s == 8 ? 0x00ff00ffu : s == 4 ? 0x0f0f0f0fu : s == 2 ? 0x33333333u
                                                                                                     : 0x55555555u;
    const uint32_t other = __shfl_xor_sync(kFull, w, s);
    w = (lane & s) ? ((w & ~low) | ((other >> s) & low)) : ((w & low) | ((other & low) << s));
  }
  return w;
}

// exclusive scan of one int per thread over the CTA; returns the prefix of this thread and the total in *total
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp /* [kRleWarps + 1] */, int* total) {
  const int lane = lane_id(), warp = warp_id();
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int up = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += up;
  }
  __syncthreads();  // s_warp may still be read from a previous scan
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < kRleWarps ? s_warp[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < kRleWarps; o <<= 1) {
      const int up = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += up;
    }
    if (lane < kRleWarps) s_warp[lane] = winc - w;
    if (lane == kRleWarps - 1) s_warp[kRleWarps] = winc;
  }
  __syncthreads();
  *total = s_warp[kRleWarps];
  return s_warp[warp] + inc - v;
}

__device__ __forceinline__ int rle_nchars(long long x) {
  int n = 0;
  bool more = true;
  while (more) {
    const int c = (int)(x & 0x1f);
    x >>= 5;
    more = (c & 0x10) ? x != -1 : x != 0;
    ++n;
  }
  return n;
}

struct RleGeom {
  const uint32_t* src;  // packed words of this mask
  int oh, ow_words, r0, r1, w0, w1, rend, n_strips;
  bool tr;              // words are stored [word][row] (word-column major) instead of [row][word]
  __device__ __forceinline__ uint32_t word(int y, int w) const {
    return __ldg(tr ? src + (size_t)w * oh + y : src + (size_t)y * ow_words + w);
  }
};

// run boundaries of the 32 columns of strip `st`, rows [r0 + 32*b, +32): returns the boundary bits of this lane's
// column (bit i = a run starts at row r0 + 32*b + i) and updates the carry (value of the pixel above the block)
__device__ __forceinline__ uint32_t rle_block_edges(const RleGeom& g, int st, int b, int lane, uint32_t& carry) {
  const int wi = g.w0 + st;
  const int y = g.r0 + 32 * b + lane;
  uint32_t word = 0;
  if (y < g.r1 && wi < g.w1) word = g.word(y, wi);
  const uint32_t col = transpose32(word, lane);
  uint32_t d = col ^ ((col << 1) | carry);
  carry = col >> 31;
  const int rows = g.rend - (g.r0 + 32 * b);  // rows of this block that exist (>= 1)
  if (rows < 32) d &= (1u << rows) - 1u;
  return d;
}

// value of the last pixel (row oh-1) of column x-1 — the pixel that precedes (x, 0) in column-major order; zero
// unless the rect reaches the bottom row and column x-1 lies inside the rect's words
__device__ __forceinline__ uint32_t rle_prev_column_last(const RleGeom& g, int x) {
  if (x == 0 || g.r1 < g.oh) return 0u;
  const int xp = x - 1, wp = xp >> 5;
  if (wp < g.w0 || wp >= g.w1) return 0u;
  return (g.word(g.oh - 1, wp) >> (xp & 31)) & 1u;
}

// value of the pixel that precedes (x, r0) in column-major order, for the first block of a column: the wrap from the
// previous column when the rect starts at row 0, otherwise the (zero) pixel above the rect
__device__ __forceinline__ uint32_t rle_first_carry(const RleGeom& g, int x) {
  return g.r0 > 0 ? 0u : rle_prev_column_last(g, x);
}

// rect reaches the bottom row but not the top one: a run that ends on the last row of column x-1 closes at (x, 0),
// a row the walk over [r0, rend) never visits.  Returns 1 if column x owes that extra boundary at position x*oh.
__device__ __forceinline__ uint32_t rle_wrap_edge(const RleGeom& g, int x) {
  return g.r0 > 0 ? rle_prev_column_last(g, x) : 0u;
}

// kSized (sized entry): the masks have the size read on the device (out of range: the count is zero, every length is
// zeroed)
template <bool kSized>
__global__ void __launch_bounds__(kRleThreads)
rle_encode_kernel(const uint32_t* __restrict__ bits_full, const int32_t* __restrict__ rect,
                  const int32_t* __restrict__ slot, const int32_t* __restrict__ count, int max_count, int oh, int ow,
                  int cap_counts, int cap_chars, uint32_t* __restrict__ counts_out, int32_t* __restrict__ n_counts,
                  uint8_t* __restrict__ chars_out, int32_t* __restrict__ n_chars, bool tr, SizedDims d) {
  chain_wait();
  if constexpr (kSized) sized_hw(d, oh, ow);
  extern __shared__ int s_col[];  // boundaries per visited column, then their exclusive prefix
  __shared__ int s_warp[kRleWarps + 1];
  const int j = blockIdx.x;
  if (j >= min(*count, max_count)) {
    if (threadIdx.x == 0) { n_counts[j] = 0; n_chars[j] = 0; }
    return;
  }
  const int k = slot ? slot[j] : j;
  const int lane = lane_id(), warp = warp_id();
  const int4 rc = reinterpret_cast<const int4*>(rect)[k];
  RleGeom g;
  g.oh = oh;
  g.tr = tr;
  g.ow_words = (ow + 31) >> 5;
  g.src = bits_full + (size_t)k * oh * g.ow_words;
  g.r0 = rc.x; g.r1 = rc.y; g.w0 = rc.z; g.w1 = rc.w;
  const bool empty = g.r1 <= g.r0 || g.w1 <= g.w0;
  if (empty) { g.r0 = g.r1 = 0; g.w0 = g.w1 = 0; }
  g.rend = min(g.r1 + 1, oh);                                 // one zero row below the rect closes the runs
  const int cend = empty ? 0 : min((g.w1 << 5) + 1, ow);      // one zero column right of the rect (wrap case)
  g.n_strips = empty ? 0 : ((cend - (g.w0 << 5)) + 31) >> 5;
  const int n_blocks = empty ? 0 : (g.rend - g.r0 + 31) >> 5;
  const int n_cols = g.n_strips << 5;
  const unsigned long long hw = (unsigned long long)oh * ow;

  // ---- pass 1: boundaries per column
  for (int st = warp; st < g.n_strips; st += kRleWarps) {
    const int x = ((g.w0 + st) << 5) + lane;
    uint32_t carry = rle_first_carry(g, x);
    int cnt = (int)rle_wrap_edge(g, x);
    for (int b = 0; b < n_blocks; ++b) {
      const uint32_t d = rle_block_edges(g, st, b, lane, carry);
      cnt += __popc(d);
    }
    s_col[(st << 5) + lane] = x < cend ? cnt : 0;
  }
  __syncthreads();
  // ---- exclusive scan over the visited columns (each thread owns a contiguous chunk)
  const int per = (n_cols + kRleThreads - 1) / kRleThreads;
  const int c_lo = min((int)threadIdx.x * per, n_cols), c_hi = min(c_lo + per, n_cols);
  int mine = 0;
  for (int c = c_lo; c < c_hi; ++c) mine += s_col[c];
  int total = 0;
  int run = block_exclusive_scan(mine, s_warp, &total);
  for (int c = c_lo; c < c_hi; ++c) {
    const int v = s_col[c];
    s_col[c] = run;
    run += v;
  }
  __syncthreads();
  const int n_edges = total;
  const int m = n_edges + 1;  // counts = differences of consecutive boundaries + the closing run
  if (m > cap_counts) {       // does not fit: report the size needed, emit nothing
    if (threadIdx.x == 0) { n_counts[j] = m; n_chars[j] = -1; }
    return;
  }
  uint32_t* cnts = counts_out + (size_t)j * cap_counts;
  // ---- pass 2: boundary positions in column-major order
  for (int st = warp; st < g.n_strips; st += kRleWarps) {
    const int x = ((g.w0 + st) << 5) + lane;
    uint32_t carry = rle_first_carry(g, x);
    int idx = s_col[(st << 5) + lane];
    if (x < cend && rle_wrap_edge(g, x)) cnts[idx++] = (uint32_t)x * (uint32_t)oh;
    for (int b = 0; b < n_blocks; ++b) {
      uint32_t d = rle_block_edges(g, st, b, lane, carry);
      if (x >= cend) d = 0;
      const uint32_t base = (uint32_t)x * (uint32_t)oh + (uint32_t)(g.r0 + 32 * b);
      while (d) {
        const int bit = __ffs(d) - 1;
        d &= d - 1;
        cnts[idx++] = base + bit;
      }
    }
  }
  __syncthreads();
  // ---- positions -> counts, in place: thread t owns [i_lo, i_hi) and reads its left neighbour before anyone writes
  const int per_m = (m + kRleThreads - 1) / kRleThreads;
  const int i_lo = min((int)threadIdx.x * per_m, m), i_hi = min(i_lo + per_m, m);
  uint32_t prev = (i_lo > 0 && i_lo < m) ? cnts[i_lo - 1] : 0u;
  __syncthreads();
  for (int i = i_lo; i < i_hi; ++i) {
    const uint32_t cur = i < n_edges ? cnts[i] : (uint32_t)hw;
    cnts[i] = cur - prev;
    prev = cur;
  }
  __syncthreads();
  // ---- string: size every count, scan, write
  int chars = 0;
  for (int i = i_lo; i < i_hi; ++i) {
    long long x = (long long)cnts[i];
    if (i > 2) x -= (long long)cnts[i - 2];
    chars += rle_nchars(x);
  }
  int total_chars = 0;
  int off = block_exclusive_scan(chars, s_warp, &total_chars);
  uint8_t* out = chars_out + (size_t)j * cap_chars;
  for (int i = i_lo; i < i_hi; ++i) {
    long long x = (long long)cnts[i];
    if (i > 2) x -= (long long)cnts[i - 2];
    bool more = true;
    while (more) {
      int c = (int)(x & 0x1f);
      x >>= 5;
      more = (c & 0x10) ? x != -1 : x != 0;
      if (more) c |= 0x20;
      if (off < cap_chars) out[off] = (uint8_t)(c + 48);
      ++off;
    }
  }
  if (threadIdx.x == 0) {
    n_counts[j] = m;
    n_chars[j] = total_chars;  // > cap_chars: the string was truncated
  }
}

int launch_rle_encode(const uint32_t* bits_full, const int32_t* rect, const int32_t* slot, const int32_t* count,
                      int max_count, int oh, int ow, int cap_counts, int cap_chars, uint32_t* counts_out,
                      int32_t* n_counts, uint8_t* chars_out, int32_t* n_chars, cudaStream_t s, bool tr,
                      const SizedDims* sized) {
  // sized (nullable): the size is read on the device; oh, ow are then the capacity (shared memory for its width)
  if (max_count <= 0) return NTTT_OK;
  if ((unsigned long long)oh * ow > 0xffffffffull) return NTTT_EUNSUPPORTED;
  const size_t smem = sizeof(int) * (size_t)(((ow + 31) / 32 + 1) * 32);
  if (smem > 160 * 1024) return NTTT_EUNSUPPORTED;
  const auto kernel = sized ? rle_encode_kernel<true> : rle_encode_kernel<false>;
  if (smem > 48 * 1024) NTTT_CUDA(set_dyn_smem(kernel, (int)smem));
  launch_chain(kernel, max_count, kRleThreads, smem, s, bits_full, rect, slot, count, max_count, oh, ow, cap_counts,
               cap_chars, counts_out, n_counts, chars_out, n_chars, tr, sized ? *sized : SizedDims{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// Packs the strings of the first n_masks outputs back to back (mask j at offset sum_{i<j} len_i) so the host reads
// sum(len) bytes instead of n_masks * max(len).  One CTA per mask; a length outside [0, cap_chars] counts as 0.
__global__ void __launch_bounds__(256)
rle_compact_kernel(const uint8_t* __restrict__ chars, const int32_t* __restrict__ n_chars, int n_masks, int cap_chars,
                   uint8_t* __restrict__ out, long long out_cap) {
  __shared__ long long s_off;
  const int j = blockIdx.x;
  if (threadIdx.x < 32) {
    long long acc = 0;
    for (int i = threadIdx.x; i < j; i += 32) {
      const int len = n_chars[i];
      acc += (len < 0 || len > cap_chars) ? 0 : len;
    }
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (threadIdx.x == 0) s_off = acc;
  }
  __syncthreads();
  int len = n_chars[j];
  if (len < 0 || len > cap_chars) len = 0;
  const long long off = s_off;
  if (off + len > out_cap) return;
  const uint8_t* src = chars + (size_t)j * cap_chars;
  uint8_t* dst = out + off;
  // (a few KB per mask and an arbitrary destination alignment: plain coalesced byte copies)
  for (int i = threadIdx.x; i < len; i += blockDim.x) dst[i] = src[i];
}

int launch_rle_compact(const uint8_t* chars, const int32_t* n_chars, int n_masks, int cap_chars, uint8_t* out,
                       long long out_cap, cudaStream_t s) {
  if (n_masks <= 0) return NTTT_OK;
  rle_compact_kernel<<<n_masks, 256, 0, s>>>(chars, n_chars, n_masks, cap_chars, out, out_cap);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
