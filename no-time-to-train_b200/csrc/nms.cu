// Class-aware box NMS on the low-res mask boxes + positive-score compaction.
//
// Reference: torchvision.ops.batched_nms(lr_bboxes.float(), pred_ious, labels, nms_thr)[:out_num]
// (Sam2MatchingBaseline_noAMG.py:621-629) and the `scores_out > 0` filter (:631-641).
// torchvision (third-party, pinned 0.19.1 by pyproject.toml:57) adds label*(max_coord+1) to every box and
// runs plain NMS; with integer-valued fp32 coordinates that is exactly "same label AND IoU > thr", which
// is what is evaluated here: inter/(areaA+areaB-inter) in fp32, areas (x2-x1)*(y2-y1), strict >.
#include "common.cuh"

namespace nttt {

// float -> uint key whose ascending order is the float's DESCENDING order (positive NaN first, like torch)
__device__ __forceinline__ uint32_t desc_key(float f) {
  uint32_t u = __float_as_uint(f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // ascending-orderable
  return ~u;
}

// single-CTA bitonic sort of (score desc, index asc); also gathers the boxes / labels into sorted order so the
// matrix kernel reads them coalesced instead of chasing order[] -> box[] pointers.
// kReg: n_pad <= 1024, one key per thread in registers (warp shuffles for the short exchanges)
template <bool kReg>
__global__ void __launch_bounds__(1024)
nms_sort_kernel(const float* __restrict__ scores, const int32_t* __restrict__ box, const int32_t* __restrict__ labels,
                int n, int n_pad, float min_score, int filter, int32_t* __restrict__ order,
                float4* __restrict__ sorted_box, int32_t* __restrict__ sorted_label, uint32_t* __restrict__ nz,
                int nz_total) {
  chain_wait();
  extern __shared__ unsigned long long s_keys[];
  // (lists above 1024 boxes) clear the per-row summary of non-zero matrix words that nms_mask_kernel ORs into
  for (int i = threadIdx.x; i < nz_total; i += blockDim.x) nz[i] = 0u;
  // filter: boxes whose score is not > min_score are not candidates at all (the reference drops them before the
  // stage, Sam2MatchingBaseline_noAMG.py:428-431): they sort last, get a unique negative label so that they never
  // match anything in the matrix, and the scan starts with them removed.
  auto make_key = [&](int i) -> unsigned long long {
    if (i >= n) return ~0ull;
    const float sc = scores[i];
    const uint32_t hi = (filter && !(sc > min_score)) ? 0xffffffffu : desc_key(sc);
    return ((unsigned long long)hi << 32) | (uint32_t)i;
  };
  auto emit = [&](int i, unsigned long long key) {
    const int o = (int)(key & 0xffffffffu);
    order[i] = o;
    const int4 bi = reinterpret_cast<const int4*>(box)[o];
    sorted_box[i] = make_float4((float)bi.x, (float)bi.y, (float)bi.z, (float)bi.w);
    sorted_label[i] = ((uint32_t)(key >> 32) == 0xffffffffu && filter) ? (-2 - i) : labels[o];
  };
  if (kReg) {
    const int i = threadIdx.x;
    unsigned long long key = make_key(i);
    key = block_bitonic_sort_1024(key, s_keys);
    if (i < n) emit(i, key);
    return;
  }
  for (int i = threadIdx.x; i < n_pad; i += blockDim.x)
    s_keys[i] = make_key(i);
  __syncthreads();
  for (int k = 2; k <= n_pad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = s_keys[i], b = s_keys[ixj];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { s_keys[i] = b; s_keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) emit(i, s_keys[i]);
}

// Long lists (n > 1024): a second order, by (label, score rank).  Class-aware suppression only acts inside a label, so in
// this order the suppression matrix is block diagonal and nms_mask_kernel skips everything else.  Single CTA, bitonic sort
// of 32-bit keys (label + bias) << 13 | score position; gathers boxes and labels into the new order and leaves the map
// class position -> score position for the scan's epilogue.
constexpr int kClassKeyBias = 8194;  // labels of filtered boxes go down to -2 - 8191
__global__ void __launch_bounds__(1024)
nms_class_sort_kernel(const float4* __restrict__ sorted_box, const int32_t* __restrict__ sorted_label, int n, int n_pad,
                      int32_t* __restrict__ c2s, float4* __restrict__ cbox, int32_t* __restrict__ clabel) {
  chain_wait();
  extern __shared__ unsigned long long s_keys[];
  uint32_t* keys = reinterpret_cast<uint32_t*>(s_keys);
  for (int i = threadIdx.x; i < n_pad; i += blockDim.x)
    keys[i] = i < n ? (((uint32_t)(sorted_label[i] + kClassKeyBias) << 13) | (uint32_t)i) : 0xffffffffu;
  __syncthreads();
  for (int k = 2; k <= n_pad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const uint32_t a = keys[i], b = keys[ixj];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int ps = (int)(keys[i] & 8191u);
    c2s[i] = ps;
    cbox[i] = sorted_box[ps];
    clabel[i] = sorted_label[ps];
  }
}

// suppression bit matrix in sorted order.  kByVictim: bit i of row j set iff i < j, same label, IoU(i,j) > thr — row j
// lists the earlier boxes that would suppress j if they are kept (wavefront scan).  Otherwise by suppressor: bit j of
// row i set iff j > i (serial scan).  The IoU arithmetic is symmetric in its two boxes (float additions commute exactly).
template <bool kByVictim>
__global__ void __launch_bounds__(256)
nms_mask_kernel(const float4* __restrict__ sorted_box, const int32_t* __restrict__ sorted_label, int n, float thr,
                uint32_t* __restrict__ mask, int row_words, uint32_t* __restrict__ nz, int nz_words, int class_sorted) {
  chain_wait();
  // class_sorted (by-victim form with the nz summary only): the boxes are ordered by (label, score) and the labels
  // ascend, so a block whose last column box has a smaller label than its first row box holds no same-label pair at all.
  // It writes nothing — the scan only reads the words flagged in `nz` — and with 80 classes that is all but the two or
  // three word tiles next to the diagonal of each row chunk.
  if (class_sorted && kByVictim) {
    const int r0 = blockIdx.y * 32, jl = min(n - 1, blockIdx.x * 256 + 255);
    if (r0 >= n || blockIdx.x * 256 > r0 + 31 || sorted_label[jl] < sorted_label[r0]) return;  // (or no column precedes a row)
  }
  __shared__ float4 s_box[8][32];
  __shared__ int s_lab[8][32];
  const int i = blockIdx.y * 32 + threadIdx.x;  // sorted position of the row box
  const int cw = blockIdx.x * 8 + threadIdx.y;  // column word
  {
    const int j = cw * 32 + threadIdx.x;
    const bool ok = j < n && cw < row_words;
    s_box[threadIdx.y][threadIdx.x] = ok ? sorted_box[j] : make_float4(0.f, 0.f, 0.f, 0.f);
    s_lab[threadIdx.y][threadIdx.x] = ok ? sorted_label[j] : -1;
  }
  __syncthreads();
  if (i >= n || cw >= row_words) return;
  uint32_t bits = 0;
  if (kByVictim ? (cw * 32 < i) : (cw * 32 + 31 > i)) {
    const float4 a = sorted_box[i];
    const float area_a = __fmul_rn(a.z - a.x, a.w - a.y);
    const int la = sorted_label[i];
    // Phase 1, branch-free: which of the 32 column boxes can suppress at all — same label, the right side of the
    // diagonal, and a non-empty intersection (inter == 0 gives ovr == 0 or 0/0 = NaN, neither is > thr >= 0).  The
    // lanes of a warp are 32 different rows, so a per-pair branch here made every warp walk the full IoU path.
    uint32_t cand = 0;
#pragma unroll 8
    for (int t = 0; t < 32; ++t) {
      const float4 b = s_box[threadIdx.y][t];
      const int j = cw * 32 + t;
      const bool side = kByVictim ? (j < i) : (j > i && j < n);
      const bool hit = side && s_lab[threadIdx.y][t] == la && fminf(a.z, b.z) > fmaxf(a.x, b.x) &&
                       fminf(a.w, b.w) > fmaxf(a.y, b.y);
      cand |= (uint32_t)hit << t;
    }
    // Phase 2: the exact fp32 IoU of torchvision's kernel on the few candidates
    const bool thr_neg = thr < 0.0f;  // (a negative threshold is also exceeded by ovr == 0: take every pair)
    if (thr_neg) cand = 0xffffffffu;
    while (cand) {
      const int t = __ffs(cand) - 1;
      cand &= cand - 1;
      const int j = cw * 32 + t;
      if ((kByVictim ? j >= i : (j <= i || j >= n)) || s_lab[threadIdx.y][t] != la) continue;
      const float4 b = s_box[threadIdx.y][t];
      const float w = fmaxf(fminf(a.z, b.z) - fmaxf(a.x, b.x), 0.0f);
      const float h = fmaxf(fminf(a.w, b.w) - fmaxf(a.y, b.y), 0.0f);
      const float inter = __fmul_rn(w, h);
      const float area_b = __fmul_rn(b.z - b.x, b.w - b.y);
      const float ovr = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
      if (ovr > thr) bits |= 1u << t;
    }
  }
  // by victim: word-major [cw][i] so that the scan's lanes (consecutive boxes) read consecutive addresses
  if (kByVictim) mask[(size_t)cw * (row_words * 32) + i] = bits;
  else mask[(size_t)i * row_words + cw] = bits;
  // which words of row i hold suppressor bits at all (class-aware NMS: very few): lets the long-list scan touch only those
  if (nz && bits) atomicOr(&nz[(size_t)i * nz_words + (cw >> 5)], 1u << (cw & 31));
}

// Greedy scan as a wavefront over 32-box chunks, one CTA of 32 warps, no CTA-wide barrier inside the scan.
// Warp c owns chunk c; lane b owns sorted box j = 32c + b and row j of the matrix (its potential
// suppressors).  keep[j] = !gone[j] && no kept suppressor:
//   * suppressors in EARLIER chunks: the lane ANDs each non-zero row word w with the final keep word K[w]; the warp waits,
//     in ascending order, on the hand-off words of exactly the chunks where ANY of its lanes has suppressor bits
//     (class-aware NMS: few) — the set is known before the first wait, and the waits are warp-uniform;
//   * suppressors in the SAME chunk: a warp-local fixed point K' = ballot(cand && !(diag & K)), which reaches the
//     unique greedy solution in (longest in-chunk chain + 1) ballots, usually 2-4 instead of a 32-step serial chain.
// Then the warp publishes K[c] together with its ready flag in one 64-bit word.  The critical path is one in-chunk
// resolve + one hand-off per chunk (measured ~1 200 cycles per hop with a flag + two block fences, ~ 300 without).  All warps of the CTA are resident and a chunk only waits on lower chunks, so the spin-waits cannot deadlock.
// Used for n <= 1024 (32 chunks = 32 warps, rows in registers); longer lists take nms_wave_sparse_kernel below.
constexpr int kScanThreads = 1024;
constexpr int kScanMaxN = 8192;

__global__ void __launch_bounds__(kScanThreads, 1)
nms_wave_kernel(const uint32_t* __restrict__ mt, int row_words, const int32_t* __restrict__ order,
                const int32_t* __restrict__ sorted_label, const float* __restrict__ top_score, int n, int max_keep,
                int32_t* __restrict__ keep, int32_t* __restrict__ n_keep, int32_t* __restrict__ sel,
                int32_t* __restrict__ n_sel) {
  chain_wait();
  __shared__ uint32_t s_K[kScanMaxN / 32];    // keep bits per chunk, then truncated to max_keep
  __shared__ uint32_t s_S[kScanMaxN / 32];    // positive-score flags, then `sel` bits
  __shared__ int s_pre[kScanMaxN / 32 + 1];   // exclusive prefix of popc over the words
  // hand-off word of a chunk: 0 until its keep bits K are final, then (1 << 32) | K.  Flag and data travel in ONE aligned
  // 64-bit shared-memory word, so neither side needs a fence (two __threadfence_block per hop made a hop ~1 200 cycles)
  __shared__ unsigned long long s_pub[32];
  volatile unsigned long long* pub = s_pub;
  const int lane = lane_id(), warp = warp_id();
  if (threadIdx.x < 32) s_pub[threadIdx.x] = 0ull;
  // n <= 1024: warp c owns chunk c, and every lane holds its whole row (<= 32 words) in registers, so no global load
  // sits on the scan's critical path
  const int c = warp;
  const int j = c * 32 + lane;
  const bool valid = j < n;
  uint32_t r[32];
#pragma unroll
  for (int w = 0; w < 32; ++w) r[w] = (valid && w <= c && w < row_words) ? __ldg(mt + (size_t)w * (row_words * 32) + j) : 0u;
  const bool gone = !valid || sorted_label[j] < -1;
  const bool pos = valid && top_score[order[valid ? j : 0]] > 0.0f;
  const uint32_t pbits = __ballot_sync(kFull, pos);
  // the earlier chunks in which ANY lane of this warp has a suppressor: the whole warp waits on exactly those, in order
  uint32_t mine = 0;
#pragma unroll
  for (int w = 0; w < 32; ++w)
    if (w < c && r[w]) mine |= 1u << w;
  const uint32_t need = __reduce_or_sync(kFull, mine);
  uint32_t own = 0;
#pragma unroll
  for (int w = 0; w < 32; ++w)
    if (w == c) own = r[w];
  const bool any_diag = __any_sync(kFull, own != 0u);  // (known before the first wait)
  __syncthreads();
  if (c < row_words) {
    uint32_t supp = 0, diag = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) {
      if (w == c) diag = r[w];  // suppressors inside this chunk (bits below the lane)
      if ((need >> w) & 1u) {   // (warp-uniform; only w < c)
        unsigned long long v;
        do { v = pub[w]; } while ((v >> 32) == 0ull);
        supp |= r[w] & (uint32_t)v;
      }
    }
    const bool cand = !gone && supp == 0;
    uint32_t K = __ballot_sync(kFull, cand);
    for (int it = 0; it < 33 && any_diag; ++it) {  // (no suppression inside the chunk: the first ballot is final)
      const uint32_t K2 = __ballot_sync(kFull, cand && (diag & K) == 0);
      if (K2 == K) break;
      K = K2;
    }
    if (lane == 0) {
      pub[c] = (1ull << 32) | K;
      s_K[c] = K;       // (read after the barrier below)
      s_S[c] = pbits;
    }
  }
  __syncthreads();
  // survivors in sorted order, truncated to max_keep; those with a positive top score also go to `sel`
  auto prefix = [&](const uint32_t* bits) {  // s_pre[w] = number of set bits in words < w (warp 0)
    if (warp == 0) {
      int run = 0;
      for (int w0 = 0; w0 < row_words; w0 += 32) {
        const int w = w0 + lane;
        const int cnt = w < row_words ? __popc(bits[w]) : 0;
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(kFull, inc, o);
          if (lane >= o) inc += up;
        }
        if (w < row_words) s_pre[w] = run + inc - cnt;
        run += __shfl_sync(kFull, inc, 31);
      }
      if (lane == 0) s_pre[row_words] = run;
    }
    __syncthreads();
  };
  prefix(s_K);
  for (int c = warp; c < row_words; c += kScanThreads / 32) {
    const uint32_t kw = s_K[c];
    const int rank = s_pre[c] + __popc(kw & ((1u << lane) - 1u));
    const bool mine = ((kw >> lane) & 1u) && rank < max_keep;
    if (mine) keep[rank] = order[c * 32 + lane];
    const uint32_t mbits = __ballot_sync(kFull, mine);
    __syncwarp();
    if (lane == 0) { s_K[c] = mbits; s_S[c] &= mbits; }
  }
  const int total_kept = min(s_pre[row_words], max_keep);
  __syncthreads();
  prefix(s_S);
  for (int c = warp; c < row_words; c += kScanThreads / 32) {
    const uint32_t sw = s_S[c];
    if ((sw >> lane) & 1u) sel[s_pre[c] + __popc(sw & ((1u << lane) - 1u))] = order[c * 32 + lane];
  }
  if (threadIdx.x == 0) { *n_keep = total_kept; *n_sel = s_pre[row_words]; }
}

// The same wavefront for lists of up to kScanMaxN boxes (points_per_side 64: 4096 candidates).  A warp owns the chunks
// c, c + 32, c + 64, ... and handles them in that order (a chunk only waits on lower chunks, which are either earlier
// rounds or lower warps of the same round, all resident: no deadlock).  A row no longer fits in registers (128 words at
// 4096 boxes), and almost all of it is zero, so the mask kernel leaves a per-row bitmap of its non-zero words (`nz`) and a
// lane loads just those — the scan's work is proportional to the suppression pairs that exist, not to n^2 / 32.
__global__ void __launch_bounds__(kScanThreads, 1)
nms_wave_sparse_kernel(const uint32_t* __restrict__ mt, const uint32_t* __restrict__ nz, int nz_words, int row_words,
                       const int32_t* __restrict__ order, const int32_t* __restrict__ sorted_label,
                       const float* __restrict__ top_score, int n, int max_keep, int32_t* __restrict__ keep,
                       int32_t* __restrict__ n_keep, int32_t* __restrict__ sel, int32_t* __restrict__ n_sel,
                       const int32_t* __restrict__ c2s) {
  // c2s (nullable): the matrix, `nz` and `sorted_label` are in CLASS order (nms_class_sort_kernel) and c2s maps a position
  // there to the box's position in score order, which is what `order` and the output lists are in: the wavefront runs in
  // class order (any order that keeps same-label boxes in score order gives the same greedy result), its keep bits are
  // scattered to score order before the compaction.
  chain_wait();
  __shared__ uint32_t s_K[kScanMaxN / 32];
  __shared__ uint32_t s_S[kScanMaxN / 32];
  __shared__ int s_pre[kScanMaxN / 32 + 1];
  __shared__ unsigned long long s_pub[kScanMaxN / 32];  // 0, then (1 << 32) | K: flag and keep bits in one word (no fences)
  volatile unsigned long long* pub = s_pub;
  const int lane = lane_id(), warp = warp_id();
  for (int i = threadIdx.x; i < row_words; i += kScanThreads) s_pub[i] = 0ull;
  __syncthreads();
  const size_t stride = (size_t)row_words * 32;
  for (int c = warp; c < row_words; c += kScanThreads / 32) {
    const int j = c * 32 + lane;
    const bool valid = j < n;
    const bool gone = !valid || sorted_label[j] < -1;
    const bool pos = valid && top_score[order[valid ? (c2s ? c2s[j] : j) : 0]] > 0.0f;
    const uint32_t pbits = __ballot_sync(kFull, pos);
    const uint32_t diag = valid ? __ldg(mt + (size_t)c * stride + j) : 0u;  // suppressors inside this chunk
    const bool any_diag = __any_sync(kFull, diag != 0u);
    uint32_t supp = 0;
    for (int q = 0; q < nz_words && q * 32 < c; ++q) {
      uint32_t m = valid ? __ldg(nz + (size_t)j * nz_words + q) : 0u;
      if (q * 32 + 32 > c) m &= (1u << (c - q * 32)) - 1u;  // words of EARLIER chunks only
      // the warp visits the union of its lanes' non-zero words in ascending order, all lanes waiting on the same
      // hand-off word; a first pass only issues the row loads so that they overlap instead of queueing behind the waits
      uint32_t all = __reduce_or_sync(kFull, m);
      uint32_t touch = 0;
      for (uint32_t t = all; t; t &= t - 1) {
        const int w = q * 32 + __ffs(t) - 1;
        if ((m >> (w & 31)) & 1u) touch |= __ldg(mt + (size_t)w * stride + j);
      }
      if (__reduce_or_sync(kFull, touch) == 0u) all = 0;  // (cannot happen: a flagged word is non-zero)
      for (; all; all &= all - 1) {
        const int w = q * 32 + __ffs(all) - 1;
        const uint32_t r = ((m >> (w & 31)) & 1u) ? __ldg(mt + (size_t)w * stride + j) : 0u;
        unsigned long long v;
        do { v = pub[w]; } while ((v >> 32) == 0ull);
        supp |= r & (uint32_t)v;
      }
    }
    const bool cand = !gone && supp == 0;
    uint32_t K = __ballot_sync(kFull, cand);
    for (int it = 0; it < 33 && any_diag; ++it) {  // (no suppression inside the chunk: the first ballot is final)
      const uint32_t K2 = __ballot_sync(kFull, cand && (diag & K) == 0);
      if (K2 == K) break;
      K = K2;
    }
    if (lane == 0) {
      pub[c] = (1ull << 32) | K;
      s_K[c] = K;  // (read after the barrier below)
      s_S[c] = pbits;
    }
  }
  __syncthreads();
  if (c2s) {  // class order -> score order (s_pub is free now: its low and high halves take the two bit vectors)
    uint32_t* k2 = reinterpret_cast<uint32_t*>(s_pub);
    uint32_t* s2 = k2 + kScanMaxN / 32;
    for (int i = threadIdx.x; i < 2 * (kScanMaxN / 32); i += kScanThreads) k2[i] = 0u;
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += kScanThreads) {
      const uint32_t kb = (s_K[j >> 5] >> (j & 31)) & 1u, sb = (s_S[j >> 5] >> (j & 31)) & 1u;
      if (kb | sb) {
        const int ps = c2s[j];
        if (kb) atomicOr(&k2[ps >> 5], 1u << (ps & 31));
        if (sb) atomicOr(&s2[ps >> 5], 1u << (ps & 31));
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < row_words; i += kScanThreads) { s_K[i] = k2[i]; s_S[i] = s2[i]; }
    __syncthreads();
  }
  auto prefix = [&](const uint32_t* bits) {  // s_pre[w] = number of set bits in words < w (warp 0)
    if (warp == 0) {
      int run = 0;
      for (int w0 = 0; w0 < row_words; w0 += 32) {
        const int w = w0 + lane;
        const int cnt = w < row_words ? __popc(bits[w]) : 0;
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(kFull, inc, o);
          if (lane >= o) inc += up;
        }
        if (w < row_words) s_pre[w] = run + inc - cnt;
        run += __shfl_sync(kFull, inc, 31);
      }
      if (lane == 0) s_pre[row_words] = run;
    }
    __syncthreads();
  };
  prefix(s_K);
  for (int c = warp; c < row_words; c += kScanThreads / 32) {
    const uint32_t kw = s_K[c];
    const int rank = s_pre[c] + __popc(kw & ((1u << lane) - 1u));
    const bool mine = ((kw >> lane) & 1u) && rank < max_keep;
    if (mine) keep[rank] = order[c * 32 + lane];
    const uint32_t mbits = __ballot_sync(kFull, mine);
    __syncwarp();
    if (lane == 0) { s_K[c] = mbits; s_S[c] &= mbits; }
  }
  const int total_kept = min(s_pre[row_words], max_keep);
  __syncthreads();
  prefix(s_S);
  for (int c = warp; c < row_words; c += kScanThreads / 32) {
    const uint32_t sw = s_S[c];
    if ((sw >> lane) & 1u) sel[s_pre[c] + __popc(sw & ((1u << lane) - 1u))] = order[c * 32 + lane];
  }
  if (threadIdx.x == 0) { *n_keep = total_kept; *n_sel = s_pre[row_words]; }
}

size_t nms_workspace_bytes(int n) {
  const size_t row_words = (size_t)ceil_div(n, 32);
  const size_t nz_words = (row_words + 31) / 32;
  return align_up(sizeof(int32_t) * (size_t)n, 256) + align_up(sizeof(uint32_t) * row_words * (row_words * 32), 256) +
         align_up(sizeof(float4) * (size_t)n, 256) + align_up(sizeof(int32_t) * (size_t)n, 256) +
         align_up(sizeof(uint32_t) * (size_t)n * nz_words, 256) +
         // class order of long lists: boxes, labels, class position -> score position
         align_up(sizeof(float4) * (size_t)n, 256) + 2 * align_up(sizeof(int32_t) * (size_t)n, 256);
}

int launch_box_nms(const int32_t* box, const float* nms_scores, const int32_t* labels, const float* top_score, int n,
                   float thr, int max_keep, int32_t* keep, int32_t* n_keep, int32_t* sel, int32_t* n_sel, void* ws,
                   size_t ws_bytes, float min_score, int filter, cudaStream_t s) {
  if (n <= 0 || max_keep <= 0) {
    NTTT_CUDA(cudaMemsetAsync(n_keep, 0, sizeof(int32_t), s));
    NTTT_CUDA(cudaMemsetAsync(n_sel, 0, sizeof(int32_t), s));
    return NTTT_OK;
  }
  if (n > kScanMaxN) return NTTT_EUNSUPPORTED;
  if (ws_bytes < nms_workspace_bytes(n)) return NTTT_EWORKSPACE;
  char* w8 = static_cast<char*>(ws);
  int32_t* order = reinterpret_cast<int32_t*>(w8);
  uint32_t* mask = reinterpret_cast<uint32_t*>(w8 + align_up(sizeof(int32_t) * (size_t)n, 256));
  const int row_words = ceil_div(n, 32);
  float4* sorted_box = reinterpret_cast<float4*>(reinterpret_cast<char*>(mask) +
                                                 align_up(sizeof(uint32_t) * (size_t)row_words * (row_words * 32), 256));
  int32_t* sorted_label = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(sorted_box) +
                                                     align_up(sizeof(float4) * (size_t)n, 256));
  const int nz_words = ceil_div(row_words, 32);
  uint32_t* nz = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(sorted_label) + align_up(sizeof(int32_t) * (size_t)n, 256));
  int n_pad = 1;
  while (n_pad < n) n_pad <<= 1;
  if (n_pad <= 1024) {
    launch_chain(nms_sort_kernel<true>, 1, 1024, sizeof(unsigned long long) * 1024, s, nms_scores, box, labels, n, 1024, min_score, filter, order,
                                                                             sorted_box, sorted_label, nullptr, 0);
  } else {
    const size_t smem = sizeof(unsigned long long) * (size_t)n_pad;
    if (smem > 48 * 1024)
      NTTT_CUDA(set_dyn_smem(nms_sort_kernel<false>, (int)smem));
    launch_chain(nms_sort_kernel<false>, 1, 1024, smem, s, nms_scores, box, labels, n, n_pad, min_score, filter, order, sorted_box,
                                                 sorted_label, nz, n * nz_words);
  }
  NTTT_LAUNCH_CHECK();
  dim3 grid(ceil_div(row_words, 8), ceil_div(n, 32));
  if (n <= 1024) {
    launch_chain(nms_mask_kernel<true>, grid, dim3(32, 8), 0, s, sorted_box, sorted_label, n, thr, mask, row_words, nullptr, 0, 0);
    NTTT_LAUNCH_CHECK();
    launch_chain(nms_wave_kernel, 1, kScanThreads, 0, s, mask, row_words, order, sorted_label, top_score, n, max_keep, keep, n_keep, sel,
                                               n_sel);
    NTTT_LAUNCH_CHECK();
    return NTTT_OK;
  }
  // longer lists: boxes re-ordered by (label, score rank), block-diagonal matrix, the same wavefront over the non-zero
  // words of each row
  float4* cbox = reinterpret_cast<float4*>(reinterpret_cast<char*>(nz) + align_up(sizeof(uint32_t) * (size_t)n * nz_words, 256));
  int32_t* clabel = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(cbox) + align_up(sizeof(float4) * (size_t)n, 256));
  int32_t* c2s = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(clabel) + align_up(sizeof(int32_t) * (size_t)n, 256));
  launch_chain(nms_class_sort_kernel, 1, 1024, sizeof(uint32_t) * (size_t)n_pad, s, sorted_box, sorted_label, n, n_pad, c2s, cbox,
               clabel);
  NTTT_LAUNCH_CHECK();
  launch_chain(nms_mask_kernel<true>, grid, dim3(32, 8), 0, s, cbox, clabel, n, thr, mask, row_words, nz, nz_words,
               /*class_sorted=*/1);
  NTTT_LAUNCH_CHECK();
  launch_chain(nms_wave_sparse_kernel, 1, kScanThreads, 0, s, mask, nz, nz_words, row_words, order, clabel, top_score, n,
               max_keep, keep, n_keep, sel, n_sel, c2s);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
