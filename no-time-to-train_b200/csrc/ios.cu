// Intersection-over-self score decay on bit-packed full-resolution masks, final top-k and output gather.
//
// Reference: obj_sim = clamp(F F^T, 0) (Sam2MatchingBaseline_noAMG.py:668-669), compute_semantic_ios
// (matching_baseline_utils.py:831-867), scores * pow(1-ios, 0.5) and argsort/top-k (:671-683).
//
// The reference casts [K,H*W] bool to fp32 and runs one SGEMM per class; the counts it produces are exact
// integers, so AND+popcount over the packed words gives the same numbers.  Only same-label pairs whose
// full-res boxes overlap can intersect, and only inside the intersection of their rects.
#include <cstdlib>

#include "common.cuh"

namespace nttt {

constexpr int kIosThreads = 256;
constexpr int kIosBigWords = 4096;  // overlap windows above this many words go to the CTA-per-pair kernel

// Pair work is symmetric (inter(i,j) and the pair similarity are shared by v_ij and v_ji), so each unordered
// same-label pair is evaluated once, by the CTA of the lower index, and both row maxima are updated with an
// integer atomicMax on the float bits (all values are >= 0).  A first tiny kernel compacts the per-mask
// metadata so the pair kernel never chases sel[] -> labels[] pointers.
struct IosMeta {
  int4 box;
  int4 rect;
  int label;
  int area;
  int src;
  int pad;
};

static size_t ios_max_pairs(int max_sel) { return (size_t)max_sel * (max_sel > 1 ? max_sel - 1 : 1) / 2 + 1; }

size_t ios_workspace_bytes(int max_sel) {
  return align_up(sizeof(IosMeta) * (size_t)max_sel, 256) + align_up(sizeof(int32_t) * (size_t)max_sel, 256) +
         align_up(sizeof(int2) * ios_max_pairs(max_sel), 256) + 256;
}

__global__ void __launch_bounds__(256)
ios_meta_kernel(const int32_t* __restrict__ rect, const int32_t* __restrict__ area_full,
                const int32_t* __restrict__ box_full, const int32_t* __restrict__ sel,
                const int32_t* __restrict__ n_sel, int max_sel, const int32_t* __restrict__ labels,
                IosMeta* __restrict__ meta, int32_t* __restrict__ label_sel, float* __restrict__ ios,
                int32_t* __restrict__ n_pairs) {
  chain_wait();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0) { n_pairs[0] = 0; n_pairs[1] = 0; }  // small list (front of the buffer), big list (back)
  if (j >= max_sel) return;
  ios[j] = 0.0f;  // identity of the row max (the zeroed diagonal, area > 0 case)
  if (j >= min(*n_sel, max_sel)) { label_sel[j] = -1; return; }
  IosMeta m;
  m.src = sel[j];
  m.label = labels[m.src];
  m.area = area_full[j];
  m.box = reinterpret_cast<const int4*>(box_full)[j];
  m.rect = reinterpret_cast<const int4*>(rect)[j];
  m.pad = 0;
  meta[j] = m;
  label_sel[j] = m.label;
}

// Pair generation: CTA i scans the partners j > i (same label, both non-empty, overlapping boxes) and appends
// (i, j) to a global list (warp-aggregated atomics).  The work per image is a few thousand pairs.
__global__ void __launch_bounds__(256)
ios_pairs_kernel(const IosMeta* __restrict__ meta, const int32_t* __restrict__ label_sel,
                 const int32_t* __restrict__ n_sel, int max_sel, int2* __restrict__ pairs,
                 int32_t* __restrict__ n_pairs, int max_pairs) {
  chain_wait();
  const int nsel = min(*n_sel, max_sel);
  const int lane = lane_id();
  for (int i = blockIdx.x; i < nsel; i += gridDim.x) {  // (row i has nsel - i - 1 partners: striding balances the CTAs)
  const IosMeta me = meta[i];
  if (me.area == 0) continue;
  for (int base = i + 1; base < nsel; base += 256) {
    const int j = base + threadIdx.x;
    bool hit = false, big = false;
    if (j < nsel && label_sel[j] == me.label) {
      const IosMeta mj = meta[j];
      const int x0 = max(me.box.x, mj.box.x), x1 = min(me.box.z, mj.box.z);
      const int y0 = max(me.box.y, mj.box.y), y1 = min(me.box.w, mj.box.w);
      hit = mj.area > 0 && x0 <= x1 && y0 <= y1;
      big = hit && ((x1 >> 5) - (x0 >> 5) + 1) * (y1 - y0 + 1) > kIosBigWords;
    }
    const uint32_t mb = __ballot_sync(kFull, big);
    const uint32_t m = __ballot_sync(kFull, hit) & ~mb;
    if (m) {
      int slot = 0;
      if (lane == 0) slot = atomicAdd(&n_pairs[0], __popc(m));
      slot = __shfl_sync(kFull, slot, 0) + __popc(m & ((1u << lane) - 1u));
      if (hit && !big) pairs[slot] = make_int2(i, j);
    }
    if (mb) {
      int slot = 0;
      if (lane == 0) slot = atomicAdd(&n_pairs[1], __popc(mb));
      slot = __shfl_sync(kFull, slot, 0) + __popc(mb & ((1u << lane) - 1u));
      if (big) pairs[max_pairs - 1 - slot] = make_int2(i, j);
    }
  }
  }
}

// The same pair generation with the metadata kernel folded in (nttt_match_image: one launch less on the chain of a single
// image).  n_pairs was zeroed by the resize kernel that ran before.  Nothing a CTA reads here is written by another CTA of
// this launch: partners are described from the raw arrays (sel -> labels, area_full, box_full), and the compacted
// records `meta[]` that the evaluation kernel reads are written on the side, each by the thread that owns the row.
__global__ void __launch_bounds__(256)
ios_pairs_fused_kernel(const int32_t* __restrict__ rect, const int32_t* __restrict__ area_full,
                       const int32_t* __restrict__ box_full, const int32_t* __restrict__ sel,
                       const int32_t* __restrict__ n_sel, int max_sel, const int32_t* __restrict__ labels,
                       IosMeta* __restrict__ meta, float* __restrict__ ios, int2* __restrict__ pairs,
                       int32_t* __restrict__ n_pairs, int max_pairs) {
  chain_wait();
  const int nsel = min(*n_sel, max_sel);
  const int lane = lane_id();
  for (int j = blockIdx.x * 256 + threadIdx.x; j < max_sel; j += gridDim.x * 256) {
    ios[j] = 0.0f;  // identity of the row max (the zeroed diagonal, area > 0 case)
    if (j < nsel) {
      IosMeta m;
      m.src = sel[j];
      m.label = labels[m.src];
      m.area = area_full[j];
      m.box = reinterpret_cast<const int4*>(box_full)[j];
      m.rect = reinterpret_cast<const int4*>(rect)[j];
      m.pad = 0;
      meta[j] = m;
    }
  }
  for (int i = blockIdx.x; i < nsel; i += gridDim.x) {  // (row i has nsel - i - 1 partners: striding balances the CTAs)
    const int my_area = area_full[i];
    if (my_area == 0) continue;
    const int my_label = labels[sel[i]];
    const int4 my_box = reinterpret_cast<const int4*>(box_full)[i];
    for (int base = i + 1; base < nsel; base += 256) {
      const int j = base + threadIdx.x;
      bool hit = false, big = false;
      if (j < nsel && labels[sel[j]] == my_label) {
        const int4 bj = reinterpret_cast<const int4*>(box_full)[j];
        const int x0 = max(my_box.x, bj.x), x1 = min(my_box.z, bj.z);
        const int y0 = max(my_box.y, bj.y), y1 = min(my_box.w, bj.w);
        hit = area_full[j] > 0 && x0 <= x1 && y0 <= y1;
        big = hit && ((x1 >> 5) - (x0 >> 5) + 1) * (y1 - y0 + 1) > kIosBigWords;
      }
      const uint32_t mb = __ballot_sync(kFull, big);
      const uint32_t m = __ballot_sync(kFull, hit) & ~mb;
      if (m) {
        int slot = 0;
        if (lane == 0) slot = atomicAdd(&n_pairs[0], __popc(m));
        slot = __shfl_sync(kFull, slot, 0) + __popc(m & ((1u << lane) - 1u));
        if (hit && !big) pairs[slot] = make_int2(i, j);
      }
      if (mb) {
        int slot = 0;
        if (lane == 0) slot = atomicAdd(&n_pairs[1], __popc(mb));
        slot = __shfl_sync(kFull, slot, 0) + __popc(mb & ((1u << lane) - 1u));
        if (big) pairs[max_pairs - 1 - slot] = make_int2(i, j);
      }
    }
  }
}

// Pairs with a LARGE overlap window (> kIosBigWords words): one CTA per pair (grid-stride over the big list, which
// grows from the back of the pair buffer): the window is spread over all threads with four load pairs in flight,
// one block reduction.  A single warp would take tens of microseconds on a 1000 x 32-word window.  Runs as the tail of
// ios_eval_kernel (every thread of the CTA arrives here): the list is usually empty, and a launch of its own put ~4 us of
// launch latency on the chain of a single image.
__device__ __forceinline__ void
ios_eval_big_pairs(const uint32_t* __restrict__ bits_full, const uint32_t* __restrict__ bits_t,
                const IosMeta* __restrict__ meta,
                const int2* __restrict__ pairs, const int32_t* __restrict__ n_pairs, int max_pairs, int max_sel, int oh,
                int ow, const float* __restrict__ obj_feats, int c, float* __restrict__ ios,
                int32_t* __restrict__ inter_out) {
  __shared__ int s_inter[kIosThreads / 32];
  __shared__ float s_dot[kIosThreads / 32];
  const int lane = lane_id(), warp = warp_id();
  constexpr int kWarps = kIosThreads / 32;
  const int ow_words = (ow + 31) >> 5;
  const int np = min(n_pairs[1], max_pairs);
  for (int p = blockIdx.x; p < np; p += gridDim.x) {
    const int2 pr = pairs[max_pairs - 1 - p];
    const int i = pr.x, j = pr.y;
    const IosMeta me = meta[i], mj = meta[j];
    const int x0 = max(me.box.x, mj.box.x), x1 = min(me.box.z, mj.box.z);
    const int y0 = max(me.box.y, mj.box.y), y1 = min(me.box.w, mj.box.w);
    const int wlo = max(max(me.rect.z, mj.rect.z), x0 >> 5), whi = min(min(me.rect.w, mj.rect.w), (x1 >> 5) + 1);
    const int ylo = max(max(me.rect.x, mj.rect.x), y0), yhi = min(min(me.rect.y, mj.rect.y), y1 + 1);
    const int nw = whi - wlo;
    const bool tr = bits_t != nullptr;  // word-column-major copy: word (y, w) at w * oh + y
    const uint32_t* mi = (tr ? bits_t : bits_full) + (size_t)i * oh * ow_words;
    const uint32_t* pj = (tr ? bits_t : bits_full) + (size_t)j * oh * ow_words;
    const size_t sy = tr ? 1 : (size_t)ow_words, sw = tr ? (size_t)oh : 1;
    int inter = 0;
    if (nw > 0 && yhi > ylo) {
      // threads tile the window: tx over words (next pow2 >= nw, <= 32), ty over rows
      int txn = 1;
      while (txn < nw && txn < 32) txn <<= 1;
      const int tx = threadIdx.x & (txn - 1), ty = threadIdx.x / txn, tyn = kIosThreads / txn;
      for (int w = wlo + tx; w < whi; w += txn) {
        int y = ylo + ty;
        for (; y + 3 * tyn < yhi; y += 4 * tyn) {
          const size_t o0 = (size_t)y * sy + (size_t)w * sw, o1 = o0 + (size_t)tyn * sy;
          const size_t o2 = o1 + (size_t)tyn * sy, o3 = o2 + (size_t)tyn * sy;
          const uint32_t a0 = __ldg(mi + o0), b0 = __ldg(pj + o0), a1 = __ldg(mi + o1), b1 = __ldg(pj + o1);
          const uint32_t a2 = __ldg(mi + o2), b2 = __ldg(pj + o2), a3 = __ldg(mi + o3), b3 = __ldg(pj + o3);
          inter += __popc(a0 & b0) + __popc(a1 & b1) + __popc(a2 & b2) + __popc(a3 & b3);
        }
        for (; y < yhi; y += tyn) {
          const size_t o = (size_t)y * sy + (size_t)w * sw;
          inter += __popc(__ldg(mi + o) & __ldg(pj + o));
        }
      }
    }
    const float* fi = obj_feats + (size_t)me.src * c;
    const float* fj = obj_feats + (size_t)mj.src * c;
    float dot = 0.0f;
    for (int e = threadIdx.x; e < c; e += kIosThreads) dot = fmaf(__ldg(fi + e), __ldg(fj + e), dot);
    inter = warp_sum(inter);
    dot = warp_sum(dot);
    if (lane == 0) { s_inter[warp] = inter; s_dot[warp] = dot; }
    __syncthreads();
    if (threadIdx.x == 0) {
      int it = 0;
      float dt = 0.0f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) { it += s_inter[w]; dt += s_dot[w]; }
      if (inter_out) {
        inter_out[(size_t)i * max_sel + j] = it;
        inter_out[(size_t)j * max_sel + i] = it;
      }
      if (it > 0) {
        const float sim = fmaxf(dt, 0.0f);
        // ((inter * s) / area) * s  — the reference's association, for both rows of the pair; all values are
        // >= 0, so the row max is an integer atomicMax on the float bits
        const float num = __fmul_rn((float)it, sim);
        atomicMax(reinterpret_cast<int*>(ios + i), __float_as_int(__fmul_rn(__fdiv_rn(num, (float)me.area), sim)));
        atomicMax(reinterpret_cast<int*>(ios + j), __float_as_int(__fmul_rn(__fdiv_rn(num, (float)mj.area), sim)));
      }
    }
    __syncthreads();
  }
}

// Pair evaluation: one WARP per pair (warp-stride over the list): popcount of the AND over the overlap window and the
// feature dot product, both reduced with shuffles — no shared memory, no CTA barrier.  (One CTA per pair spent most of
// its instructions on per-thread set-up and the block reduction: a typical window is ~150 words.)  A window is walked
// row-major with the lanes along the words when it is wide and along the rows when it is narrow.
// bits_t (nullable): the word-column-major copy [k][word][row] written by upsample_pack2_kernel.  A window is a few words
// wide and hundreds of rows tall: in the row-major layout every word sits in its own 32-byte sector (ncu: 80 MB through L1
// for 10 MB of words); in the column-major copy a warp reads 128 contiguous bytes per word column.
// kSized (sized entry): the packed masks have the size read on the device (out of range: the pair list is empty).
template <bool kSized>
__global__ void __launch_bounds__(kIosThreads)
ios_eval_kernel(const uint32_t* __restrict__ bits_full, const uint32_t* __restrict__ bits_t,
                const IosMeta* __restrict__ meta,
                const int2* __restrict__ pairs, const int32_t* __restrict__ n_pairs, int max_pairs, int max_sel, int oh,
                int ow, const float* __restrict__ obj_feats, int c, float* __restrict__ ios,
                int32_t* __restrict__ inter_out, SizedDims d) {
  chain_wait();
  if constexpr (kSized) sized_hw(d, oh, ow);
  const int lane = lane_id();
  constexpr int kWarps = kIosThreads / 32;
  const int ow_words = (ow + 31) >> 5;
  const int np = min(*n_pairs, max_pairs);
  const uint32_t mask_words = (uint32_t)oh * (uint32_t)ow_words;
  for (int p = blockIdx.x * kWarps + warp_id(); p < np; p += gridDim.x * kWarps) {
    const int2 pr = pairs[p];
    const int i = pr.x, j = pr.y;
    const IosMeta me = meta[i], mj = meta[j];
    const int x0 = max(me.box.x, mj.box.x), x1 = min(me.box.z, mj.box.z);
    const int y0 = max(me.box.y, mj.box.y), y1 = min(me.box.w, mj.box.w);
    const int wlo = max(max(me.rect.z, mj.rect.z), x0 >> 5), whi = min(min(me.rect.w, mj.rect.w), (x1 >> 5) + 1);
    const int ylo = max(max(me.rect.x, mj.rect.x), y0), yhi = min(min(me.rect.y, mj.rect.y), y1 + 1);
    const int nw = whi - wlo, nr = yhi - ylo;
    const uint32_t* mi = bits_full + (size_t)i * mask_words;
    const uint32_t* pj = bits_full + (size_t)j * mask_words;
    int inter = 0;
    if (bits_t && nw > 0 && nr > 0) {
      // column-major copy: lanes along the rows of one word column, four row chunks in flight
      const uint32_t* ti = bits_t + (size_t)i * mask_words;
      const uint32_t* tj = bits_t + (size_t)j * mask_words;
      for (int w = wlo; w < whi; ++w) {
        const uint32_t base = (uint32_t)w * (uint32_t)oh;
        int y = ylo + lane;
        for (; y + 96 < yhi; y += 128) {
          const uint32_t a0 = __ldg(ti + base + y), b0 = __ldg(tj + base + y);
          const uint32_t a1 = __ldg(ti + base + y + 32), b1 = __ldg(tj + base + y + 32);
          const uint32_t a2 = __ldg(ti + base + y + 64), b2 = __ldg(tj + base + y + 64);
          const uint32_t a3 = __ldg(ti + base + y + 96), b3 = __ldg(tj + base + y + 96);
          inter += __popc(a0 & b0) + __popc(a1 & b1) + __popc(a2 & b2) + __popc(a3 & b3);
        }
        for (; y < yhi; y += 32) inter += __popc(__ldg(ti + base + y) & __ldg(tj + base + y));
      }
    } else if (nw > 0 && nr > 0) {
      // lanes tile the window: tx over words (next pow2 >= nw, <= 32), ty over rows
      int txn = 1;
      while (txn < nw && txn < 32) txn <<= 1;
      const int tx = lane & (txn - 1), ty = lane / txn, tyn = 32 / txn;
      for (int w = wlo + tx; w < whi; w += txn) {
        uint32_t o = (uint32_t)(ylo + ty) * (uint32_t)ow_words + (uint32_t)w;
        const uint32_t step = (uint32_t)tyn * (uint32_t)ow_words;
        int y = ylo + ty;
        for (; y + 3 * tyn < yhi; y += 4 * tyn, o += 4 * step) {
          const uint32_t a0 = __ldg(mi + o), b0 = __ldg(pj + o), a1 = __ldg(mi + o + step), b1 = __ldg(pj + o + step);
          const uint32_t a2 = __ldg(mi + o + 2 * step), b2 = __ldg(pj + o + 2 * step);
          const uint32_t a3 = __ldg(mi + o + 3 * step), b3 = __ldg(pj + o + 3 * step);
          inter += __popc(a0 & b0) + __popc(a1 & b1) + __popc(a2 & b2) + __popc(a3 & b3);
        }
        for (; y < yhi; y += tyn, o += step) inter += __popc(__ldg(mi + o) & __ldg(pj + o));
      }
    }
    inter = warp_sum(inter);
    if (inter_out && lane == 0) {
      inter_out[(size_t)i * max_sel + j] = inter;
      inter_out[(size_t)j * max_sel + i] = inter;
    }
    if (inter > 0) {  // (warp-uniform) the similarity is only needed for intersecting pairs
      const float* fi = obj_feats + (size_t)me.src * c;
      const float* fj = obj_feats + (size_t)mj.src * c;
      float dot = 0.0f;
      if ((c & 3) == 0) {
        const float4* f4i = reinterpret_cast<const float4*>(fi);
        const float4* f4j = reinterpret_cast<const float4*>(fj);
        for (int e = lane; e < (c >> 2); e += 32) {
          const float4 a = __ldg(f4i + e), b = __ldg(f4j + e);
          dot = fmaf(a.x, b.x, dot); dot = fmaf(a.y, b.y, dot); dot = fmaf(a.z, b.z, dot); dot = fmaf(a.w, b.w, dot);
        }
      } else {
        for (int e = lane; e < c; e += 32) dot = fmaf(__ldg(fi + e), __ldg(fj + e), dot);
      }
      dot = warp_sum(dot);
      if (lane == 0) {
        const float sim = fmaxf(dot, 0.0f);
        // ((inter * s) / area) * s  — the reference's association, for both rows of the pair; all values are
        // >= 0, so the row max is an integer atomicMax on the float bits
        const float num = __fmul_rn((float)inter, sim);
        atomicMax(reinterpret_cast<int*>(ios + i), __float_as_int(__fmul_rn(__fdiv_rn(num, (float)me.area), sim)));
        atomicMax(reinterpret_cast<int*>(ios + j), __float_as_int(__fmul_rn(__fdiv_rn(num, (float)mj.area), sim)));
      }
    }
  }
  ios_eval_big_pairs(bits_full, bits_t, meta, pairs, n_pairs, max_pairs, max_sel, oh, ow, obj_feats, c, ios, inter_out);
}

// rows of empty full-res masks: 0/0 on the diagonal -> NaN, and torch.max propagates it
__global__ void __launch_bounds__(256)
ios_finalize_kernel(const int32_t* __restrict__ area_full, const int32_t* __restrict__ n_sel, int max_sel,
                    float* __restrict__ ios) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < min(*n_sel, max_sel) && area_full[j] == 0) ios[j] = __int_as_float(0x7fc00000);
}

// the two pair counters inside the workspace (small list, big list)
int32_t* ios_pair_counters(void* ws, int max_sel) {
  char* w8 = static_cast<char*>(ws);
  char* pairs = w8 + align_up(sizeof(IosMeta) * (size_t)max_sel, 256) + align_up(sizeof(int32_t) * (size_t)max_sel, 256);
  return reinterpret_cast<int32_t*>(pairs + align_up(sizeof(int2) * ios_max_pairs(max_sel), 256));
}

// finalize=false leaves the NaN rows to the consumer (decay_rank_kernel applies the same rule)
int launch_mask_ios(const uint32_t* bits_full, const int32_t* rect, const int32_t* area_full, const int32_t* box_full,
                    const int32_t* sel, const int32_t* n_sel, int max_sel, int oh, int ow, const int32_t* labels,
                    const float* obj_feats, int c, float* ios, int32_t* inter_out, void* ws, bool finalize,
                    cudaStream_t s, const uint32_t* bits_t, bool counters_zeroed, const SizedDims* sized) {
  // sized (nullable): the size of the packed masks is read on the device; oh, ow are then the capacity
  // counters_zeroed: the pair counters (ios_pair_counters(ws, max_sel)) were set to zero by an earlier kernel of the
  // same stream — the metadata kernel is then folded into the pair kernel
  if (max_sel <= 0) return NTTT_OK;
  if (inter_out) NTTT_CUDA(cudaMemsetAsync(inter_out, 0, sizeof(int32_t) * (size_t)max_sel * max_sel, s));
  char* w8 = static_cast<char*>(ws);
  IosMeta* meta = reinterpret_cast<IosMeta*>(w8);
  int32_t* label_sel = reinterpret_cast<int32_t*>(w8 + align_up(sizeof(IosMeta) * (size_t)max_sel, 256));
  int2* pairs = reinterpret_cast<int2*>(reinterpret_cast<char*>(label_sel) + align_up(sizeof(int32_t) * (size_t)max_sel, 256));
  const int max_pairs = (int)ios_max_pairs(max_sel);
  int32_t* n_pairs = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(pairs) + align_up(sizeof(int2) * (size_t)max_pairs, 256));
  const int pair_grid = t_low_latency ? max_sel : min(max_sel, 148);
  if (counters_zeroed) {
    launch_chain(ios_pairs_fused_kernel, pair_grid, 256, 0, s, rect, area_full, box_full, sel, n_sel, max_sel, labels, meta, ios,
                 pairs, n_pairs, max_pairs);
    NTTT_LAUNCH_CHECK();
  } else {
    launch_chain(ios_meta_kernel, ceil_div(max_sel, 256), 256, 0, s, rect, area_full, box_full, sel, n_sel, max_sel, labels, meta,
                 label_sel, ios, n_pairs);
    NTTT_LAUNCH_CHECK();
    launch_chain(ios_pairs_kernel, pair_grid, 256, 0, s, meta, label_sel, n_sel, max_sel, pairs, n_pairs, max_pairs);
    NTTT_LAUNCH_CHECK();
  }
  // one CTA per SM when many images are in flight (measured 89.4 vs 90.0 us/image with four), four for one image alone
  launch_chain(sized ? ios_eval_kernel<true> : ios_eval_kernel<false>, t_low_latency ? 148 * 4 : 148, kIosThreads, 0, s,
               bits_full, bits_t, meta, pairs, n_pairs, max_pairs, max_sel, oh, ow, obj_feats, c, ios, inter_out,
               sized ? *sized : SizedDims{});
  NTTT_LAUNCH_CHECK();
  if (finalize) {
    ios_finalize_kernel<<<ceil_div(max_sel, 256), 256, 0, s>>>(area_full, n_sel, max_sel, ios);
    NTTT_LAUNCH_CHECK();
  }
  return NTTT_OK;
}

// ---------------------------------------------------------------------------------------------------
// decay + final ranking: decayed = score * sqrt(1 - ios); order = argsort(desc), NaN first, stable.
// Single CTA bitonic sort on (key, position) over <= 1024 entries (max_sel <= 8*num_out_instance).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t desc_key_nanfirst(float f) {
  if (f != f) return 0u;  // every NaN first
  uint32_t u = __float_as_uint(f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  u = ~u;
  return u == 0u ? 1u : u;  // keep 0 reserved for NaN (only +NaN patterns could map to 0 anyway)
}

__global__ void __launch_bounds__(1024)
decay_rank_kernel(const float* __restrict__ top_score, const int32_t* __restrict__ labels,
                  const float* __restrict__ ios, const int32_t* __restrict__ sel, const int32_t* __restrict__ n_sel,
                  int max_sel, int n_pad, int num_out, const int32_t* __restrict__ box_full,
                  const int32_t* __restrict__ area_full,
                  int64_t* __restrict__ out_boxes, float* __restrict__ out_scores, int64_t* __restrict__ out_labels,
                  int32_t* __restrict__ out_index, int32_t* __restrict__ out_slot, int32_t* __restrict__ n_out,
                  float* __restrict__ decayed_out) {
  chain_wait();
  extern __shared__ unsigned long long s_keys[];
  float* s_val = reinterpret_cast<float*>(s_keys + n_pad);
  const int nsel = min(*n_sel, max_sel);
  auto make_key = [&](int i) -> unsigned long long {
    if (i >= nsel) return ~0ull;
    // empty full-res mask: the reference's 0/0 on the IoS diagonal -> NaN (torch.max propagates it)
    const float io = (area_full && area_full[i] == 0) ? __int_as_float(0x7fc00000) : ios[i];
    const float d = __fmul_rn(top_score[sel[i]], sqrtf(__fsub_rn(1.0f, io)));
    s_val[i] = d;
    if (decayed_out) decayed_out[i] = d;
    return ((unsigned long long)desc_key_nanfirst(d) << 32) | (uint32_t)i;
  };
  if (n_pad <= 1024) {
    // one key per thread, warp shuffles for the short exchanges (n_pad == 1024 by construction of the launcher)
    unsigned long long key = make_key(threadIdx.x);
    __syncthreads();  // s_val complete before s_keys is reused as the exchange buffer? (distinct regions) - keep order
    key = block_bitonic_sort_1024(key, s_keys);
    s_keys[threadIdx.x] = key;
    __syncthreads();
  } else {
    for (int i = threadIdx.x; i < n_pad; i += blockDim.x) s_keys[i] = make_key(i);
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
  }
  const int nout = min(num_out, nsel);
  for (int r = threadIdx.x; r < nout; r += blockDim.x) {
    const int k = (int)(s_keys[r] & 0xffffffffu);  // slot in the selected list
    const int src = sel[k];
    out_slot[r] = k;
    out_index[r] = src;
    out_scores[r] = s_val[k];
    out_labels[r] = (int64_t)labels[src];
    const int4 b = reinterpret_cast<const int4*>(box_full)[k];
    out_boxes[4 * r + 0] = b.x; out_boxes[4 * r + 1] = b.y; out_boxes[4 * r + 2] = b.z; out_boxes[4 * r + 3] = b.w;
  }
  if (threadIdx.x == 0) *n_out = nout;
}

int launch_decay_rank(const float* top_score, const int32_t* labels, const float* ios, const int32_t* sel,
                      const int32_t* n_sel, int max_sel, int num_out, const int32_t* box_full,
                      const int32_t* area_full, int64_t* out_boxes,
                      float* out_scores, int64_t* out_labels, int32_t* out_index, int32_t* out_slot, int32_t* n_out,
                      float* decayed_out, cudaStream_t s) {
  if (max_sel <= 0 || num_out <= 0) {
    NTTT_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int32_t), s));
    return NTTT_OK;
  }
  int n_pad = 1024;  // the register sort always runs the 1024-key network
  while (n_pad < max_sel) n_pad <<= 1;
  const size_t smem = (sizeof(unsigned long long) + sizeof(float)) * (size_t)n_pad;
  if (smem > 200 * 1024) return NTTT_EUNSUPPORTED;
  if (smem > 48 * 1024)
    NTTT_CUDA(set_dyn_smem(decay_rank_kernel, (int)smem));
  launch_chain(decay_rank_kernel, 1, 1024, smem, s, top_score, labels, ios, sel, n_sel, max_sel, n_pad, num_out, box_full,
                                          area_full, out_boxes, out_scores, out_labels, out_index, out_slot, n_out, decayed_out);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
