// Full-resolution mask pass: antialiased bilinear resize of the selected low-res logits to the original
// image size, strict > 0, bit-pack, area and box — without materialising the fp32 [K,H,W] tensor.
//
// Reference: Sam2MatchingBaseline_noAMG.py:657-665 (F.interpolate(..., antialias=True) > 0,
// batched_mask_to_box).  Arithmetic: horizontal pass on each contributing input row, then vertical
// pass, each `acc = s0*w0; acc = fma(s_j, w_j, acc)` in fp32 — the association of aten's
// upsample_gen2d_aa kernel (ATen/native/cuda/UpSample.cuh interpolate_aa_single_dim).
//
// Two exact shortcuts keep the kernel off the instruction roofline:
//   1. rect bound: an output sample whose footprint lies outside the low-res box sees only
//      non-positive logits and non-negative weights, so it is not > 0.  Only the rect is computed/stored.
//   2. uniform footprints: if every low-res bit under the footprint of a 32-pixel output word is 0 the
//      word is 0; if every bit is 1 (and the mask's positives are finite, flags bit0) the word is all
//      ones.  Only words whose footprint crosses the mask boundary evaluate the interpolation.
#include "common.cuh"

namespace nttt {

constexpr int kUpThreads = 128;
constexpr int kUpMaxSplit = 8;       // grid.x: CTAs available per mask; a mask uses ceil(groups / kUpGroupsPerCta) of them
constexpr int kUpCols = 8;           // word columns per group slot of a warp
constexpr int kUpSub = 32 / kUpCols;  // group slots per warp
constexpr int kUpGroupsPerCta = 32;  // row groups per CTA = 8 per warp: amortises the per-CTA / per-warp set-up

struct UpTables {
  const int32_t* xmin; const int32_t* xsize; const float* wx; int tx;
  const int32_t* ymin; const int32_t* ysize; const float* wy; int ty;
  const int32_t* x_tlo; const int32_t* x_tlen;  // input col -> output range
  const int32_t* y_tlo; const int32_t* y_tlen;  // input row -> output range
  const int32_t* y_grp_of; const int32_t* y_grp_start;  // output rows grouped by identical input span
  // two-tap records (every span <= 2 input samples: up-scaling), else nullptr: {min | size << 16} and {w0, w1}
  const uint32_t* pkx_span; const float2* pkx_w; const uint32_t* pky_span; const float2* pky_w;
};

// acc = s0*w0; acc = fma(s_j, w_j, acc)
__device__ __forceinline__ float aa_dot(const float* __restrict__ src, int stride, const float* __restrict__ w, int n) {
  float acc = __fmul_rn(__ldg(src), __ldg(w));
  for (int j = 1; j < n; ++j) acc = __fmaf_rn(__ldg(src + (size_t)j * stride), __ldg(w + j), acc);
  return acc;
}

// scratch per mask (zero-initialised by the meta kernel): {area, maxx+1, maxy+1, BIG-minx, BIG-miny, done}
constexpr int kScratchInts = 8;
constexpr int kBig = 1 << 30;
constexpr int kTapsReg = 4;  // footprints of up to 4 input rows keep their horizontal-pass values in registers

// per selected mask, resolved once by a tiny pre-kernel so that the CTAs of a mask do not each chase
// sel[] -> box_lr[] -> span tables; scratch[kScratchInts*k + 6..7] is unused padding
struct alignas(16) UpMeta {  // 48 bytes: three 128-bit loads
  const float* logits;  // the candidate's [ih, iw] logits
  int src;              // index into bits_lr / box_lr (candidate number)
  int safe;             // flags bit0
  int r0, r1;           // output rows [r0, r1)
  int w0, w1;           // output words [w0, w1)
  int lr0, lr1;         // low-res rows [lr0, lr1) under those output rows
  int g0, g1;           // row groups [g0, g1) covering [r0, r1)
};

// Sized entry (nttt_match_image_sized): the kSized instance of each resize kernel reads the output size (h, w) from
// device memory when it runs and takes the tables of the context's atlas entry of that size instead of the (oh, ow, t)
// it was launched with.  The first kernel of the first resize chain also writes the status (counts[3]) and, for a size
// outside the range, empties the selection (counts[1] = 0) so that every later kernel sees no work.  A chain whose path
// (two-tap or general) the size does not take exits here, as does every resize kernel for a size outside the range.
__device__ __forceinline__ bool sized_tables(const SizedDims& d, bool two_tap, bool status, int& oh, int& ow,
                                             UpTables& t) {
  const bool in_range = sized_hw(d, oh, ow);
  if (status && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    d.counts[3] = in_range ? 0 : 1;
    if (!in_range) d.counts[1] = 0;
  }
  if (!in_range) return false;
  const SizedAxis y = d.ay[oh - d.min_h], x = d.ax[ow - d.min_w];
  if ((x.pk_span != nullptr && y.pk_span != nullptr) != two_tap) return false;
  t = UpTables{x.xmin, x.xsize, x.w, x.taps, y.xmin, y.xsize, y.w, y.taps, x.t_lo, x.t_len, y.t_lo, y.t_len,
               y.grp_of, y.grp_start, x.pk_span, x.pk_w, y.pk_span, y.pk_w};
  return true;
}

// (A function of its own: written inside the kernel, these statements compile to different SASS; this is the one
// measured.)
__device__ __forceinline__ void
upsample_meta_body(const uint32_t* __restrict__ bits_lr, const int32_t* __restrict__ box_lr,
                   const int32_t* __restrict__ flags_lr, int ih, int iw, const int32_t* __restrict__ sel,
                   const int32_t* __restrict__ n_sel, int max_sel, const UpTables& t, UpMeta* __restrict__ meta,
                   int32_t* __restrict__ rect, int32_t* __restrict__ scratch, const float* __restrict__ logits,
                   const float* const* __restrict__ mask_ptr) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= max_sel) return;
#pragma unroll
  for (int q = 0; q < kScratchInts; ++q) scratch[(size_t)k * kScratchInts + q] = 0;
  if (k >= min(*n_sel, max_sel)) return;
  UpMeta m;
  m.src = sel[k];
  m.logits = mask_ptr ? mask_ptr[m.src] : logits + (size_t)m.src * ih * iw;
  const int4 b = reinterpret_cast<const int4*>(box_lr)[m.src];
  // empty low-res mask <=> box all zero AND bit (0,0) clear
  const bool lr_empty = (b.x | b.y | b.z | b.w) == 0 && (bits_lr[(size_t)m.src * ih * (iw >> 5)] & 1u) == 0;
  m.r0 = m.r1 = m.w0 = m.w1 = m.lr0 = m.lr1 = m.g0 = m.g1 = 0;
  if (!lr_empty) {
    m.r0 = t.y_tlo[b.y];
    m.r1 = t.y_tlo[b.w] + t.y_tlen[b.w];
    const int c0 = t.x_tlo[b.x];
    const int c1 = t.x_tlo[b.z] + t.x_tlen[b.z];
    m.w0 = c0 >> 5;
    m.w1 = (c1 + 31) >> 5;
    if (m.r1 > m.r0) {
      m.lr0 = t.ymin[m.r0];
      m.lr1 = t.ymin[m.r1 - 1] + t.ysize[m.r1 - 1];
      m.g0 = t.y_grp_of[m.r0];
      m.g1 = t.y_grp_of[m.r1 - 1] + 1;
    }
  }
  m.safe = flags_lr[m.src] & 1;
  meta[k] = m;
  reinterpret_cast<int4*>(rect)[k] = make_int4(m.r0, m.r1, m.w0, m.w1);
}

template <bool kSized>
__global__ void __launch_bounds__(256)
upsample_meta_kernel(const uint32_t* __restrict__ bits_lr, const int32_t* __restrict__ box_lr,
                     const int32_t* __restrict__ flags_lr, int ih, int iw, const int32_t* __restrict__ sel,
                     const int32_t* __restrict__ n_sel, int max_sel, UpTables t, UpMeta* __restrict__ meta,
                     int32_t* __restrict__ rect, int32_t* __restrict__ scratch, const float* __restrict__ logits,
                     const float* const* __restrict__ mask_ptr, SizedDims d) {
  if constexpr (kSized) {
    int oh, ow;
    if (!sized_tables(d, false, true, oh, ow, t)) return;
  }
  upsample_meta_body(bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, t, meta, rect, scratch, logits, mask_ptr);
}

__device__ __forceinline__ int up_ctas_needed(int n_groups) {
  return max(1, min(kUpMaxSplit, (n_groups + kUpGroupsPerCta - 1) / kUpGroupsPerCta));
}

// grid (kUpMaxSplit, max_sel).  A mask with G row groups is served by ceil(G / 32) CTAs (the others exit at once); a
// CTA (4 warps) takes 32 consecutive groups, warp w the groups w, w+4, ... of them, FOUR at a time: lane = (group slot,
// word column), 8 columns per slot (wider masks loop over column chunks).  Per group: the footprint test on the low-res
// bits (shared memory) classifies each word as all-0, all-1 or mixed; mixed words are evaluated one at a time by the
// whole warp with lane = pixel (the owning lane broadcasts its group's rows): horizontal pass of the shared input rows
// once, vertical pass per output row, one ballot per row.
// All indices inside the loops are 32-bit (one 64-bit base per array): 64-bit index arithmetic was a third of the
// instructions of an earlier version.
// Logit tile staging: the taps of every boundary word of a CTA lie in the low-res rows [clr0, clr1) x the columns under
// the mask's output words.  Read one by one from global memory they are chains of dependent DRAM accesses (pk_x record
// -> logits -> pk_y record) and the kernel sat at 18 % issue utilisation; instead the CTA copies that tile into shared
// memory once with 16-byte cp.async (no register is held while the copies are in flight, rows are contiguous
// segments: full sectors, each logit of the box read at most once per CTA) and the evaluation reads LDS.
// `stage_floats` = capacity of the tile area in floats (0: staging off); tiles that do not fit (very wide / tall
// chunks, more than 256 row groups) and the configurations without two-tap records take the direct path, which stays
// bit-identical.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <bool kSized>
__global__ void __launch_bounds__(kUpThreads, 5)
upsample_pack_kernel(const uint32_t* __restrict__ bits_lr, const UpMeta* __restrict__ meta, int ih, int iw,
                     const int32_t* __restrict__ n_sel, int max_sel, int oh, int ow, UpTables t,
                     uint32_t* __restrict__ bits_full, int32_t* __restrict__ area_full, int32_t* __restrict__ box_full,
                     int32_t* __restrict__ scratch, int stage_floats, SizedDims d) {
  if constexpr (kSized) {
    if (!sized_tables(d, false, false, oh, ow, t)) return;
  }
  extern __shared__ __align__(16) uint32_t s_lr[];  // packed low-res bits of this mask, rows [clr0, clr1) only; then the tile
  __shared__ int s_red[5];
  const int k = blockIdx.y;
  if (k >= min(*n_sel, max_sel)) return;
  const UpMeta mt = meta[k];
  const int n_groups = mt.g1 - mt.g0;
  const int needed = up_ctas_needed(n_groups);
  if ((int)blockIdx.x >= needed) return;
  const int lr_wpr = iw >> 5;
  const int ow_words = (ow + 31) >> 5;
  const int lane = lane_id(), warp = warp_id();
  constexpr int kWarps = kUpThreads / 32;
  const int r0 = mt.r0, r1 = mt.r1, w0 = mt.w0, w1 = mt.w1;
  const int chunk0 = mt.g0 + blockIdx.x * kUpGroupsPerCta;       // first group of this CTA's first chunk
  const bool one_chunk = needed * kUpGroupsPerCta >= n_groups;   // (false only beyond 256 groups)

  // low-res rows under this CTA's groups
  int clr0 = mt.lr0, clr1 = mt.lr1;
  if (one_chunk && chunk0 < mt.g1) {
    const int gl = min(chunk0 + kUpGroupsPerCta, mt.g1);
    const int ya = max(t.y_grp_start[chunk0], r0), yb = min(t.y_grp_start[gl], r1);
    clr0 = t.ymin[ya];
    clr1 = t.ymin[yb - 1] + t.ysize[yb - 1];
  }
  const uint32_t* lr = bits_lr + ((size_t)mt.src * ih + clr0) * lr_wpr;
  const int n_lr = (clr1 - clr0) * lr_wpr;
  const bool fast_cfg = t.pkx_span != nullptr && t.pky_span != nullptr;  // <= 2 taps on both axes
  const float* src = mt.logits;
  // tile = low-res rows [clr0, clr1) x columns [tc0, tc0 + tstride) (4-float aligned), behind the bits (16-byte aligned)
  float* tile = reinterpret_cast<float*>(s_lr + (((ih * lr_wpr + 1) + 3) & ~3));
  int tc0 = 0, tstride = 0;
  bool staged = false;
  if (fast_cfg && one_chunk && chunk0 < mt.g1 && stage_floats > 0 && w1 > w0) {
    const int xa = min(w0 << 5, ow - 1), xb = min((w1 << 5) - 1, ow - 1);
    tc0 = t.xmin[xa] & ~3;
    tstride = min((t.xmin[xb] + t.xsize[xb] + 3) & ~3, iw) - tc0;
    staged = tstride > 0 && (clr1 - clr0) * tstride <= stage_floats;
  }
  if (staged) {
    const int cpr = tstride >> 2;  // 16-byte chunks per tile row
    const int n_chunks = (clr1 - clr0) * cpr;
    const float* g0p = src + (size_t)clr0 * iw + tc0;
    for (int i = threadIdx.x; i < n_chunks; i += kUpThreads) {
      const int row = i / cpr, c4 = (i - row * cpr) << 2;
      cp_async16(tile + row * tstride + c4, g0p + (size_t)row * iw + c4);
    }
  }
  for (int i = threadIdx.x; i < n_lr; i += kUpThreads) s_lr[i] = lr[i];
  if (threadIdx.x < 5) s_red[threadIdx.x] = 0;
  const bool safe = mt.safe != 0;
  // taps are read at  tap_base[row * tap_stride + col - tap_c0]  (generic loads: global logits or the shared tile)
  const float* tap_base = staged ? tile - clr0 * tstride : src;
  const int tap_stride = staged ? tstride : iw;
  const int tap_c0 = staged ? tc0 : 0;
  uint32_t* dst = bits_full + (size_t)k * oh * ow_words;
  cp_async_wait_all();
  __syncthreads();

  int area = 0, minx = kBig, maxx = -1, miny = kBig, maxy = -1;
  // A warp works on kUpSub row groups at once: lane = (group slot q, word column): a mask is ~7 words wide, so with one
  // group per warp three lanes in four idled through the per-group part (spans, footprint test, stores, statistics),
  // which was as many instructions as the evaluation of the boundary words itself.
  const int q = lane / kUpCols;
  for (int wbase = w0; wbase < w1; wbase += kUpCols) {
    // per-lane (= per output word) constants, hoisted out of the row-group loop
    const int wi = wbase + (lane & (kUpCols - 1));
    const bool active = wi < w1;
    const int x0 = min(wi << 5, ow - 1);
    const int x1 = min(x0 + 31, ow - 1);
    const uint32_t valid = (x1 - x0 == 31) ? 0xffffffffu : ((1u << (x1 - x0 + 1)) - 1u);
    const int c0 = t.xmin[x0];
    const int c1 = t.xmin[x1] + t.xsize[x1];  // exclusive
    const int cw0 = c0 >> 5;
    const bool two_words = ((c1 - 1) >> 5) <= cw0 + 1;  // the footprint columns span at most two low-res words
    uint32_t m0, m1 = 0;
    {
      const int lo = c0 - (cw0 << 5), hi = min(c1 - (cw0 << 5), 32);
      m0 = (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
      const int hi1 = c1 - ((cw0 + 1) << 5);
      if (hi1 > 0) m1 = hi1 >= 32 ? 0xffffffffu : ((1u << hi1) - 1u);
    }
    uint32_t colbits = 0;
    for (int cb = chunk0; cb < mt.g1; cb += needed * kUpGroupsPerCta) {
      const int cend = min(cb + kUpGroupsPerCta, mt.g1);
      for (int g0 = cb + warp; g0 < cend; g0 += kWarps * kUpSub) {
        const int g = g0 + kWarps * q;
        const bool gvalid = g < cend;
        // rows [ya, yb) of this group share the input rows [ry0, ry0 + rys)   (no group: ya = yb = r0, nrows = 0)
        const int ya = gvalid ? max(t.y_grp_start[g], r0) : r0, yb = gvalid ? min(t.y_grp_start[g + 1], r1) : r0;
        const int nrows = yb - ya;
        int ry0, rys;
        if (fast_cfg) {
          const int pky = (int)__ldg(t.pky_span + (uint32_t)ya);
          ry0 = pky & 0xffff;
          rys = pky >> 16;
        } else {
          ry0 = t.ymin[ya];
          rys = t.ysize[ya];
        }
        const int rb = ry0 * tap_stride - tap_c0;    // index of the group's first input row at column 0
        const int lrb = (ry0 - clr0) * lr_wpr + cw0;  // this lane's first footprint word in s_lr
        uint32_t words[kGrpMax];
#pragma unroll
        for (int j = 0; j < kGrpMax; ++j) words[j] = 0;
        bool mixed = false;
        if (active && gvalid) {
          bool all0 = true, all1 = true;
          if (two_words) {
            // (m1 == 0 when the footprint stays inside one low-res word; s_lr has a spare word at the end)
            uint32_t any = 0, miss = 0;
            if (rys <= 3) {
#pragma unroll
              for (int r = 0; r < 3; ++r) {
                if (r < rys) {
                  const uint32_t v0 = s_lr[(uint32_t)(lrb + r * lr_wpr)] & m0;
                  const uint32_t v1 = s_lr[(uint32_t)(lrb + r * lr_wpr + 1)] & m1;
                  any |= v0 | v1;
                  miss |= (v0 ^ m0) | (v1 ^ m1);
                }
              }
            } else {
              for (int r = 0; r < rys; ++r) {
                const uint32_t v0 = s_lr[lrb + r * lr_wpr] & m0;
                const uint32_t v1 = s_lr[lrb + r * lr_wpr + 1] & m1;
                any |= v0 | v1;
                miss |= (v0 ^ m0) | (v1 ^ m1);
              }
            }
            all0 = any == 0;
            all1 = miss == 0;
          } else {
            for (int r = 0; r < rys; ++r) {
              const uint32_t* row = s_lr + (lrb - cw0) + r * lr_wpr;
              for (int cw = cw0; cw <= (c1 - 1) >> 5; ++cw) {
                const int lo = max(c0 - (cw << 5), 0), hi = min(c1 - (cw << 5), 32);
                const uint32_t m = (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
                const uint32_t v = row[cw] & m;
                all0 = all0 && (v == 0);
                all1 = all1 && (v == m);
              }
            }
          }
          if (all1 && safe && !all0) {
#pragma unroll
            for (int j = 0; j < kGrpMax; ++j) words[j] = valid;
          } else if (!all0) {
            mixed = true;
          }
        }
        uint32_t todo = __ballot_sync(kFull, mixed);
        while (todo) {
          const int src_lane = __ffs(todo) - 1;
          todo &= todo - 1;
          // the word's group: its rows and input rows come from the lane that owns the word
          const int s_ya = __shfl_sync(kFull, ya, src_lane), s_nrows = __shfl_sync(kFull, nrows, src_lane);
          const int s_rb = __shfl_sync(kFull, rb, src_lane), s_rys = __shfl_sync(kFull, rys, src_lane);
          const int x = ((wbase + (src_lane & (kUpCols - 1))) << 5) + lane;
          if (fast_cfg) {
            // The pixel's span and two weights (records past the width have size 0).  Taps beyond the span are never
            // read; rows / taps beyond it contribute fma(0, 0, acc) = acc, so the arithmetic is exactly
            // acc = s0*w0; acc = fma(s_j, w_j, acc) for j < size, horizontally and then vertically.
            const float2 xt = __ldg(t.pkx_w + (uint32_t)x);
            const int pk = (int)__ldg(t.pkx_span + (uint32_t)x);
            const int cx = pk & 0xffff, cs = pk >> 16;
            float T[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              float acc = 0.0f;
              if (r < s_rys) {  // (warp-uniform)
                // records past the image width have cs = 0, cx = 0 and zero weights: their first tap is clamped to
                // the first column of the row (a valid address) and the lane's result is masked by `cs > 0`
                const float* pl = tap_base + (s_rb + max(cx, tap_c0) + r * tap_stride);
                acc = __fmul_rn(*pl, xt.x);
                if (cs > 1) acc = __fmaf_rn(pl[1], xt.y, acc);
              }
              T[r] = acc;
            }
#pragma unroll
            for (int j = 0; j < kGrpMax; ++j) {
              // {w0, w1} of the group's rows (rows past its last one repeat it and are dropped at the store)
              const float2 wv = __ldg(t.pky_w + (uint32_t)min(s_ya + j, s_ya + s_nrows - 1));
              float acc = __fmul_rn(T[0], wv.x);
              acc = __fmaf_rn(T[1], wv.y, acc);
              const uint32_t res = __ballot_sync(kFull, cs > 0 && acc > 0.0f);
              if (lane == src_lane) words[j] = res;
            }
            continue;
          }
          const bool inb = x < ow;
          const int cx = inb ? t.xmin[x] : 0, cs = inb ? t.xsize[x] : 1;
          const float* wx = t.wx + (size_t)(inb ? x : 0) * t.tx;
          const float* p = src + (s_rb + cx);  // (never staged here: tap_stride == iw, tap_c0 == 0)
          if (s_rys <= kTapsReg) {
            // horizontal pass once per group, vertical pass per row
            float T[kTapsReg];
#pragma unroll
            for (int r = 0; r < kTapsReg; ++r) T[r] = (r < s_rys && inb) ? aa_dot(p + (size_t)r * iw, 1, wx, cs) : 0.0f;
#pragma unroll
            for (int j = 0; j < kGrpMax; ++j) {
              if (j < s_nrows) {
                const float* wy = t.wy + (size_t)(s_ya + j) * t.ty;
                float acc = __fmul_rn(T[0], __ldg(wy));
#pragma unroll
                for (int r = 1; r < kTapsReg; ++r)
                  if (r < s_rys) acc = __fmaf_rn(T[r], __ldg(wy + r), acc);
                const uint32_t res = __ballot_sync(kFull, inb && acc > 0.0f);
                if (lane == src_lane) words[j] = res;
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < kGrpMax; ++j) {
              if (j < s_nrows) {
                const float* wy = t.wy + (size_t)(s_ya + j) * t.ty;
                float acc = 0.0f;
                if (inb) {
                  acc = __fmul_rn(aa_dot(p, 1, wx, cs), __ldg(wy));
                  for (int r = 1; r < s_rys; ++r) acc = __fmaf_rn(aa_dot(p + (size_t)r * iw, 1, wx, cs), __ldg(wy + r), acc);
                }
                const uint32_t res = __ballot_sync(kFull, inb && acc > 0.0f);
                if (lane == src_lane) words[j] = res;
              }
            }
          }
        }
        // store + statistics (words[] is zero on inactive lanes and on rows that were not computed)
        const int doff = ya * ow_words + wi;
#pragma unroll
        for (int j = 0; j < kGrpMax; ++j) {
          const uint32_t word = j < nrows ? words[j] : 0u;  // (the fast path computes all kGrpMax rows)
          if (active && j < nrows) dst[(uint32_t)(doff + j * ow_words)] = word;
          area += __popc(word);
          colbits |= word;
          if (word) {
            miny = min(miny, ya + j);
            maxy = max(maxy, ya + j);
          }
        }
      }
    }
    if (colbits) {
      minx = min(minx, (wi << 5) + __ffs(colbits) - 1);
      maxx = max(maxx, (wi << 5) + 31 - __clz(colbits));
    }
  }
  area = warp_sum(area);
  minx = warp_min(minx); miny = warp_min(miny); maxx = warp_max(maxx); maxy = warp_max(maxy);
  if (lane == 0) {
    atomicAdd(&s_red[0], area);
    atomicMax(&s_red[1], maxx + 1);
    atomicMax(&s_red[2], maxy + 1);
    atomicMax(&s_red[3], kBig - minx);
    atomicMax(&s_red[4], kBig - miny);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int32_t* sc = scratch + (size_t)k * kScratchInts;
    atomicAdd(&sc[0], s_red[0]);
    atomicMax(&sc[1], s_red[1]);
    atomicMax(&sc[2], s_red[2]);
    atomicMax(&sc[3], s_red[3]);
    atomicMax(&sc[4], s_red[4]);
    __threadfence();
    const int prev = atomicAdd(&sc[5], 1);
    if (prev == needed - 1) {  // last CTA of this mask publishes the final statistics
      __threadfence();
      const int a = atomicAdd(&sc[0], 0);
      const int mx1 = atomicMax(&sc[1], 0), my1 = atomicMax(&sc[2], 0);
      const int bx = atomicMax(&sc[3], 0), by = atomicMax(&sc[4], 0);
      area_full[k] = a;
      int4 o = make_int4(0, 0, 0, 0);
      if (a > 0) o = make_int4(kBig - bx, kBig - by, mx1 - 1, my1 - 1);
      reinterpret_cast<int4*>(box_full)[k] = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// v2 — the path every two-tap configuration takes (every span of both axes <= 2 samples: up-scaling, see
// aa_spans_within_two)
//
// What v1 measured as (ncu, config 2): 18-33 % issue utilisation, top stall long-scoreboard on the chain
// pk_x record -> logits -> pk_y record, 4 800 of 6 400 CTAs exiting after two dependent global loads, ~165 warp
// instructions per boundary word.  v2 changes the organisation, not the arithmetic:
//   * a PLAN kernel turns the selected masks into a compact list of work items (mask, 32 row groups, 8 word columns)
//     with their geometry resolved; persistent CTAs pull items from it with one atomic — no empty CTAs;
//   * everything an item reads is copied into shared memory up front with cp.async (no register held while in flight):
//     the logit tile under its rows/columns, the packed low-res rows, the two-tap x / y records, the group boundaries.
//     The evaluation loop then has no global load at all;
//   * a warp owns a word COLUMN of the item: lane = row group for the footprint classification (32 groups at once),
//     lane = pixel for the evaluation, so the pixel's x record is loaded once per column instead of once per word and
//     group data are warp-uniform shared-memory reads instead of shuffles;
//   * results go to a shared-memory tile; the epilogue writes them out in 32-byte row segments and derives area and box
//     from the words (no per-row statistics inside the loops).
// ---------------------------------------------------------------------------------------------------
constexpr int kUp2Threads = 128;
constexpr int kUp2Groups = 32;                       // row groups per item = lanes of the classification
constexpr int kUp2Cols = 8;                          // word columns per item
constexpr int kUp2Rows = kUp2Groups * kGrpMax;       // output rows per item (<= 128)
constexpr int kUp2OutStride = kUp2Rows + kUp2Rows / 32;  // column-major result tile, one pad word per 32 rows
constexpr int kUp2CtasPerSm = 7;

struct alignas(16) Up2Item {  // 32 bytes, written by the plan kernel
  int k;                 // selected-mask slot
  int g;                 // first group | n_groups << 16
  int w;                 // first word  | n_words  << 16
  int y;                 // first output row | n_rows << 16
  int lr;                // first low-res row | n_lr_rows << 16
  int tc;                // first tile column (multiple of 4) | tile stride << 16
  int staged;            // 1: the logit tile fits the shared-memory budget
  int pad;
};

// A few CTAs (gridDim.x = P), no table staging, no atomics.  Per strip of 1024 masks EVERY CTA resolves the geometry of
// every mask of the strip (four per thread, all loads read-only so that they overlap) and runs the same block scan of the
// item counts — a few hundred redundant table reads are cheaper than a cross-CTA scan or a counter that somebody has to
// zero — and then writes its share of the item records (item e belongs to CTA e mod P ... in blocks of 256): thread per ITEM,
// the mask found by binary search over the offsets.  CTA (k / 256) mod P owns the per-mask outputs (meta, rect, scratch).
// The single-CTA form of this kernel spent 18 us on ~7 dependent access rounds of 1024 threads each; this one is a
// handful of L2 round trips long.  ctr[0] = number of items, ctr[1] = next item to hand out (zeroed for the main kernel).
constexpr int kPlanThreads = 256;
constexpr int kPlanPerThread = 1024 / kPlanThreads;

// floats of the logit tile: what an item needs at the size (`need`, see up2_tile_factor), bounded by the staging budget
__host__ __device__ __forceinline__ int up2_tile_floats(long need, int stage_floats) {
  int floats = (int)(need < stage_floats ? need : stage_floats);
  if (floats < 0) floats = 0;
  return (floats + 3) & ~3;
}

// (A function of its own: written inside the kernel, these statements compile to different SASS; this is the one
// measured.)
__device__ __forceinline__ void
upsample_plan_body(const uint32_t* __restrict__ bits_lr, const int32_t* __restrict__ box_lr,
                   const int32_t* __restrict__ flags_lr, int ih, int iw, const int32_t* __restrict__ sel,
                   const int32_t* __restrict__ n_sel, int max_sel, const UpTables& t, UpMeta* __restrict__ meta,
                   int32_t* __restrict__ rect, int32_t* __restrict__ scratch, const float* __restrict__ logits,
                   const float* const* __restrict__ mask_ptr, Up2Item* __restrict__ items, int32_t* __restrict__ ctr,
                   int32_t* __restrict__ area_full, int32_t* __restrict__ box_full, int oh, int ow, int tile_cap_floats) {
  __shared__ int s_warp[kPlanThreads / 32 + 1];
  __shared__ int s_off[1024];   // exclusive item offset of each mask of the strip
  __shared__ int s_ccs[1024];   // column chunks of each mask (0: no items)
  __shared__ int4 s_geo[1024];  // {g0, g1, w0, w1} of each mask of the strip
  __shared__ int2 s_rows[1024]; // {r0, r1}
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(__ldg(n_sel), max_sel);
  const int words_lr = ih * (iw >> 5);
  int base = 0;
  for (int k0 = 0; k0 < max_sel; k0 += 1024) {
    // ---- geometry of masks k0 + tid * kPlanPerThread + q (consecutive masks per thread: the scan below is then a
    //      thread-local prefix + one block scan of the thread totals)
    int cnt[kPlanPerThread];
    int thread_items = 0;
#pragma unroll
    for (int q = 0; q < kPlanPerThread; ++q) {
      const int idx = tid * kPlanPerThread + q;
      const int k = k0 + idx;
      const bool owner = ((k >> 8) % gridDim.x) == blockIdx.x;
      int n_items = 0, ccs = 0;
      int4 geo = make_int4(0, 0, 0, 0);
      int2 rows = make_int2(0, 0);
      if (k < max_sel && owner) {
#pragma unroll
        for (int z = 0; z < kScratchInts; ++z) scratch[(size_t)k * kScratchInts + z] = 0;
      }
      if (k < n) {
        UpMeta m;
        m.r0 = m.r1 = m.w0 = m.w1 = m.lr0 = m.lr1 = m.g0 = m.g1 = 0;
        m.src = __ldg(sel + k);
        m.logits = mask_ptr ? mask_ptr[m.src] : logits + (size_t)m.src * ih * iw;
        const int4 b = __ldg(reinterpret_cast<const int4*>(box_lr) + m.src);
        const bool lr_empty = (b.x | b.y | b.z | b.w) == 0 && (__ldg(bits_lr + (size_t)m.src * words_lr) & 1u) == 0;
        if (!lr_empty) {
          m.r0 = __ldg(t.y_tlo + b.y);
          m.r1 = __ldg(t.y_tlo + b.w) + __ldg(t.y_tlen + b.w);
          const int c0 = __ldg(t.x_tlo + b.x);
          const int c1 = __ldg(t.x_tlo + b.z) + __ldg(t.x_tlen + b.z);
          m.w0 = c0 >> 5;
          m.w1 = (c1 + 31) >> 5;
          if (m.r1 > m.r0) {
            m.lr0 = __ldg(t.ymin + m.r0);
            m.lr1 = __ldg(t.ymin + m.r1 - 1) + __ldg(t.ysize + m.r1 - 1);
            m.g0 = __ldg(t.y_grp_of + m.r0);
            m.g1 = __ldg(t.y_grp_of + m.r1 - 1) + 1;
          }
        }
        m.safe = __ldg(flags_lr + m.src) & 1;
        geo = make_int4(m.g0, m.g1, m.w0, m.w1);
        rows = make_int2(m.r0, m.r1);
        const bool has = m.r1 > m.r0 && m.w1 > m.w0;
        if (has) {
          ccs = (m.w1 - m.w0 + kUp2Cols - 1) / kUp2Cols;
          n_items = ((m.g1 - m.g0 + kUp2Groups - 1) / kUp2Groups) * ccs;
        }
        if (owner) {
          meta[k] = m;
          reinterpret_cast<int4*>(rect)[k] = make_int4(m.r0, m.r1, m.w0, m.w1);
          if (has) {
            scratch[(size_t)k * kScratchInts + 6] = n_items;
          } else {  // nothing to compute: publish the empty result here
            area_full[k] = 0;
            reinterpret_cast<int4*>(box_full)[k] = make_int4(0, 0, 0, 0);
          }
        }
      }
      cnt[q] = n_items;
      thread_items += n_items;
      s_ccs[idx] = ccs;
      s_geo[idx] = geo;
      s_rows[idx] = rows;
    }
    // ---- exclusive scan of the item counts over the strip
    int inc = thread_items;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += up;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const int w = lane < kPlanThreads / 32 ? s_warp[lane] : 0;
      int winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, winc, o);
        if (lane >= o) winc += up;
      }
      __syncwarp();
      if (lane < kPlanThreads / 32) s_warp[lane] = winc - w;
      if (lane == 31) s_warp[kPlanThreads / 32] = winc;
    }
    __syncthreads();
    {
      int off = s_warp[warp] + inc - thread_items;
#pragma unroll
      for (int q = 0; q < kPlanPerThread; ++q) {
        s_off[tid * kPlanPerThread + q] = off;
        off += cnt[q];
      }
    }
    __syncthreads();
    const int strip_items = s_warp[kPlanThreads / 32];
    // ---- item records: blocks of kPlanThreads consecutive items go round-robin over the CTAs
    for (int e = blockIdx.x * kPlanThreads + tid; e < strip_items; e += gridDim.x * kPlanThreads) {
      // last mask of the strip whose offset is <= e: masks without items share the offset of their successor, so the
      // LAST of equal offsets is the one that owns the item
      int lo = 0, hi = 1023;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_off[mid] <= e) lo = mid; else hi = mid - 1;
      }
      const int4 g = s_geo[lo];
      const int2 r = s_rows[lo];
      const int i = e - s_off[lo], cc_n = s_ccs[lo];
      const int rc = i / cc_n, cc = i - rc * cc_n;
      const int gA = g.x + rc * kUp2Groups, gB = min(gA + kUp2Groups, g.y);
      const int wA = g.z + cc * kUp2Cols, wB = min(wA + kUp2Cols, g.w);
      const int ya = min(max(__ldg(t.y_grp_start + gA), r.x), r.y), yb = min(max(__ldg(t.y_grp_start + gB), r.x), r.y);
      const int l0 = __ldg(t.ymin + ya), l1 = __ldg(t.ymin + yb - 1) + __ldg(t.ysize + yb - 1);
      const int xa = min(wA << 5, ow - 1), xb = min((wB << 5) - 1, ow - 1);
      const int tc0 = __ldg(t.xmin + xa) & ~3;
      const int tstride = min((__ldg(t.xmin + xb) + __ldg(t.xsize + xb) + 3) & ~3, iw) - tc0;
      Up2Item it;
      it.k = k0 + lo;
      it.g = gA | ((gB - gA) << 16);
      it.w = wA | ((wB - wA) << 16);
      it.y = ya | ((yb - ya) << 16);
      it.lr = l0 | ((l1 - l0) << 16);
      it.tc = tc0 | (tstride << 16);
      it.staged = (l1 - l0) * tstride <= tile_cap_floats ? 1 : 0;
      it.pad = 0;
      items[base + e] = it;
    }
    base += strip_items;
    __syncthreads();  // the strip's shared arrays are rewritten by the next strip
  }
  if (blockIdx.x == 0 && tid == 0) { ctr[0] = base; ctr[1] = 0; }
}

// tile_cap_floats: the tile budget of the size.  The kSized instance derives it on the device from the size's budget
// factors, bounded by stage_floats (the context's staging budget) as launch_upsample_pack does for a static size;
// status: this is the first kernel of the sized entry's resize.
template <bool kSized>
__global__ void __launch_bounds__(kPlanThreads)
upsample_plan_kernel(const uint32_t* __restrict__ bits_lr, const int32_t* __restrict__ box_lr,
                     const int32_t* __restrict__ flags_lr, int ih, int iw, const int32_t* __restrict__ sel,
                     const int32_t* __restrict__ n_sel, int max_sel, UpTables t, UpMeta* __restrict__ meta,
                     int32_t* __restrict__ rect, int32_t* __restrict__ scratch, const float* __restrict__ logits,
                     const float* const* __restrict__ mask_ptr, Up2Item* __restrict__ items, int32_t* __restrict__ ctr,
                     int32_t* __restrict__ area_full, int32_t* __restrict__ box_full, int oh, int ow, int tile_cap_floats,
                     int stage_floats, bool status, SizedDims d) {
  chain_wait();
  if constexpr (kSized) {
    if (!sized_tables(d, true, status, oh, ow, t)) return;
    tile_cap_floats = up2_tile_floats((long)d.ay[oh - d.min_h].budget * (long)d.ax[ow - d.min_w].budget, stage_floats);
  }
  upsample_plan_body(bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, t, meta, rect, scratch, logits, mask_ptr,
                     items, ctr, area_full, box_full, oh, ow, tile_cap_floats);
}

// 16-byte copy that allocates in L1: the two-tap records are a few KB shared by every item an SM processes
__device__ __forceinline__ void cp_async16_ca(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t saddr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr));
  return v;
}

// Two taps per axis.  aten's kernel runs `acc = s0*w0; acc = fma(s_j, w_j, acc)` over the table's taps; with up-scaling
// every span has <= 2 samples, so a third term is always fma(0, 0, acc) = acc + 0.  That is acc itself for every acc
// (inf and NaN included) except -0, which becomes +0, and a zero's sign never decides `acc > 0` (neither zero passes,
// and a later non-zero term swamps it), so leaving those terms out keeps every thresholded bit.  A second tap beyond
// the span (size 1) still enters as fma(0, 0, acc): its value is not read (the neighbour may be inf or NaN).

// taps of one input row for this lane's pixel
template <bool kStaged>
__device__ __forceinline__ float up2_row(const float* __restrict__ gsrc, uint32_t saddr, int idx, const float2& wx, int cs) {
  float a0, a1 = 0.0f;
  if (kStaged) {
    const uint32_t p = saddr + ((uint32_t)idx << 2);
    a0 = lds_f32(p);
    if (cs > 1) a1 = lds_f32(p + 4);
  } else {
    const float* p = gsrc + idx;
    a0 = __ldg(p);
    if (cs > 1) a1 = __ldg(p + 1);
  }
  return __fmaf_rn(a1, wx.y, __fmul_rn(a0, wx.x));
}

// per-group record of an item (shared memory): output row offset, rows, first tile row index * stride, input rows
struct alignas(16) Up2Group { int row, nrows, trow, rys; };

template <bool kStaged>
__device__ __forceinline__ void up2_evaluate(int warp, int lane, int n_list, const uint16_t* __restrict__ s_list,
                                             const Up2Group* __restrict__ s_grp, const uint32_t* __restrict__ s_xspan,
                                             const float2* __restrict__ s_xw, const float2* __restrict__ s_yw,
                                             uint32_t* __restrict__ s_out, const float* __restrict__ gsrc,
                                             uint32_t tile_saddr, int tap_stride, int tap_c0) {
  constexpr int kWarps = kUp2Threads / 32;
  for (int e = warp; e < n_list; e += kWarps) {
    const int ent = s_list[e];
    const int u = ent >> 5, gl = ent & 31;
    const Up2Group g = s_grp[gl];
    const int px = (u << 5) + lane;
    const int pk = (int)s_xspan[px];
    const float2 wx = s_xw[px];
    const int cx = pk & 0xffff, cs = pk >> 16;  // records past the image width: cs = 0, cx = 0, zero weights
    const int idx = g.trow + max(cx - tap_c0, 0);
    // horizontal pass of the group's (<= 2) input rows.  A group with one input row (image border) reads its row twice
    // and takes 0 for the second: no branch, and the second row's weight is 0.
    const float T0 = up2_row<kStaged>(gsrc, tile_saddr, idx, wx, cs);
    const float T1r = up2_row<kStaged>(gsrc, tile_saddr, idx + (g.rys > 1 ? tap_stride : 0), wx, cs);
    const float T1 = g.rys > 1 ? T1r : 0.0f;
    // vertical pass, all kGrpMax rows: rows past the group's last one read the records that follow and are dropped at
    // the store.  Nearly every group is full when up-scaling (groups are runs of equal spans), and a per-row branch
    // around the ballot costs more issue slots than the row itself.
    const float2* wy = s_yw + g.row;
    uint32_t mine = 0;
#pragma unroll
    for (int j = 0; j < kGrpMax; ++j) {
      const float2 wv = wy[j];
      const float acc = __fmaf_rn(T1, wv.y, __fmul_rn(T0, wv.x));
      const uint32_t res = __ballot_sync(kFull, cs > 0 && acc > 0.0f);
      if (lane == j) mine = res;
    }
    if (lane < g.nrows) {
      const int row = g.row + lane;
      s_out[u * kUp2OutStride + row + (row >> 5)] = mine;
    }
  }
}

// one item's area / box into its mask's scratch; the last item of the mask publishes the mask's totals
__device__ __forceinline__ void up2_publish(int k, const int (&red)[5], int32_t* __restrict__ scratch,
                                            int32_t* __restrict__ area_full, int32_t* __restrict__ box_full) {
  int32_t* sc = scratch + (size_t)k * kScratchInts;
  atomicAdd(&sc[0], red[0]);
  atomicMax(&sc[1], red[1]);
  atomicMax(&sc[2], red[2]);
  atomicMax(&sc[3], red[3]);
  atomicMax(&sc[4], red[4]);
  __threadfence();
  const int prev = atomicAdd(&sc[5], 1);
  if (prev == sc[6] - 1) {  // last item of this mask
    __threadfence();
    const int a = atomicAdd(&sc[0], 0);
    const int mx1 = atomicMax(&sc[1], 0), my1 = atomicMax(&sc[2], 0);
    const int bx = atomicMax(&sc[3], 0), by = atomicMax(&sc[4], 0);
    area_full[k] = a;
    int4 o = make_int4(0, 0, 0, 0);
    if (a > 0) o = make_int4(kBig - bx, kBig - by, mx1 - 1, my1 - 1);
    reinterpret_cast<int4*>(box_full)[k] = o;
  }
}

template <bool kSized>
__global__ void __launch_bounds__(kUp2Threads, kUp2CtasPerSm)
upsample_pack2_kernel(const uint32_t* __restrict__ bits_lr, const UpMeta* __restrict__ meta, int ih, int iw, int oh,
                      int ow, UpTables t, uint32_t* __restrict__ bits_full, uint32_t* __restrict__ bits_t,
                      int32_t* __restrict__ area_full, int32_t* __restrict__ box_full, int32_t* __restrict__ scratch,
                      const Up2Item* __restrict__ items, int32_t* __restrict__ ctr, int32_t* __restrict__ zero2,
                      SizedDims d) {
  chain_wait();
  // (nullable) two counters of the NEXT stage, zeroed here so that its first kernel can append to them right away (also
  // for a size out of range)
  if (zero2 && blockIdx.x == 0 && threadIdx.x == 0) { zero2[0] = 0; zero2[1] = 0; }
  if constexpr (kSized) {
    if (!sized_tables(d, true, false, oh, ow, t)) return;
  }
  extern __shared__ __align__(16) unsigned char s_raw[];
  // two-tap records of the item's columns and rows; the rows from ya0 rounded down to a multiple of 4 (16-byte copies)
  float2* s_xw = reinterpret_cast<float2*>(s_raw);                        // [kUp2Cols * 32]
  float2* s_yw = s_xw + kUp2Cols * 32;                                    // [kUp2Rows + 8] (3 rows past the end are read)
  uint32_t* s_xspan = reinterpret_cast<uint32_t*>(s_yw + kUp2Rows + 8);   // [kUp2Cols * 32]
  uint32_t* s_yspan = s_xspan + kUp2Cols * 32;                            // [kUp2Rows + 4]
  Up2Group* s_grp = reinterpret_cast<Up2Group*>(s_yspan + kUp2Rows + 4);  // [kUp2Groups]
  uint32_t* s_out = reinterpret_cast<uint32_t*>(s_grp + kUp2Groups);      // [kUp2Cols * kUp2OutStride]
  int* s_gstart = reinterpret_cast<int*>(s_out + kUp2Cols * kUp2OutStride);  // [kUp2Groups + 4]
  uint16_t* s_list = reinterpret_cast<uint16_t*>(s_gstart + kUp2Groups + 4);  // [kUp2Cols * kUp2Groups] boundary words
  const int lr_wpr = iw >> 5;
  uint32_t* s_lr = reinterpret_cast<uint32_t*>(s_list + kUp2Cols * kUp2Groups);  // [ih * lr_wpr + 4] (one spare word is read)
  float* tile = reinterpret_cast<float*>(s_lr + ((ih * lr_wpr + 4 + 3) & ~3));
  __shared__ int s_item;
  __shared__ int s_red[5];
  __shared__ uint32_t s_mix[kUp2Cols];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kUp2Threads / 32;
  const int ow_words = (ow + 31) >> 5;
  const int total = ctr[0];
  const uint32_t tile_saddr = (uint32_t)__cvta_generic_to_shared(tile);
  // Thread 0 claims the next item while the current one runs, and publishes an item's statistics while the next one's
  // copies are in flight: the round trips of those atomics and of the fence no longer hold the whole CTA.
  int next = 0, pend_k = -1, pend[5];
  if (tid == 0) s_item = atomicAdd(&ctr[1], 1);
  for (;;) {
    __syncthreads();  // the previous item is completely done with shared memory; s_item is the claimed item
    const int item = s_item;
    if (item >= total) break;
    if (tid == 0) next = atomicAdd(&ctr[1], 1);
    if (tid < 5) s_red[tid] = 0;
    const Up2Item it = items[item];
    const int k = it.k;
    const UpMeta mt = meta[k];
    const int gA = it.g & 0xffff, ng = it.g >> 16;
    const int wA = it.w & 0xffff, nw = it.w >> 16;
    const int ya0 = it.y & 0xffff, n_rows = it.y >> 16;
    const int clr0 = it.lr & 0xffff, tr = it.lr >> 16;
    const int tc0 = it.tc & 0xffff, tstride = it.tc >> 16;
    const bool staged = it.staged != 0;
    const float* src = mt.logits;
    // ---- stage everything the item reads (cp.async: nothing is held in registers while in flight)
    if (staged) {
      const int cpr = tstride >> 2;  // 16-byte chunks per tile row
      // one warp per row, lanes along its 16-byte chunks; source pointer and shared address advance by constants
      // (the indexed form spent ~20 instructions per row on address arithmetic: 8 % of this kernel)
      const float* gp = src + (size_t)(clr0 + warp) * iw + tc0 + (lane << 2);
      uint32_t sp = tile_saddr + (uint32_t)((warp * tstride + (lane << 2)) << 2);
      const uint32_t sp_step = (uint32_t)(kWarps * tstride) << 2;
      const size_t gp_step = (size_t)kWarps * iw;
      for (int row = warp; row < tr; row += kWarps, gp += gp_step, sp += sp_step)
        for (int c = lane; c < cpr; c += 32)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sp + ((uint32_t)(c - lane) << 4)), "l"(gp + ((c - lane) << 2)) : "memory");
    }
    {
      const uint32_t* lr = bits_lr + ((size_t)mt.src * ih + clr0) * lr_wpr;
      const int n_lr = tr * lr_wpr;
      // (rows of iw / 32 words: 16-byte chunks when the row length allows, which every multiple of 128 pixels does)
      if ((lr_wpr & 3) == 0 && (reinterpret_cast<uintptr_t>(lr) & 15) == 0) {
        for (int i = tid; i < (n_lr >> 2); i += kUp2Threads) cp_async16_ca(s_lr + 4 * i, lr + 4 * i);
      } else {
        for (int i = tid; i < n_lr; i += kUp2Threads) cp_async4(s_lr + i, lr + i);
      }
      // (the tables are padded to a multiple of 32 coordinates: the rounded-up ends stay inside them)
      const int yb = ya0 & ~3, ny = n_rows + (ya0 & 3);
      for (int i = tid; i < ((ny + 3) >> 2); i += kUp2Threads) cp_async16_ca(s_yspan + 4 * i, t.pky_span + yb + 4 * i);
      for (int i = tid; i < ((ny + 1) >> 1); i += kUp2Threads) cp_async16_ca(s_yw + 2 * i, t.pky_w + yb + 2 * i);
      for (int i = tid; i < (nw << 3); i += kUp2Threads) cp_async16_ca(s_xspan + 4 * i, t.pkx_span + (wA << 5) + 4 * i);
      for (int i = tid; i < (nw << 4); i += kUp2Threads) cp_async16_ca(s_xw + 2 * i, t.pkx_w + (wA << 5) + 2 * i);
      if (tid <= ng) s_gstart[tid] = min(max(t.y_grp_start[gA + tid], mt.r0), mt.r1);
    }
    if (tid == 0 && pend_k >= 0) up2_publish(pend_k, pend, scratch, area_full, box_full);
    cp_async_wait_all();
    __syncthreads();
    // taps are read at index  trow + max(col - tap_c0, 0)  of the shared tile (staged) or of the global logits
    const int tap_stride = staged ? tstride : iw;
    const int tap_c0 = staged ? tc0 : 0;
    const bool safe = mt.safe != 0;
    // ---- phase A: footprint classification, lane = row group, warp w takes the columns w, w + 4
    int my_ya = 0, my_nrows = 0, my_ry0 = 0, my_rys = 0;
    if (lane < ng) {
      my_ya = s_gstart[lane];
      my_nrows = s_gstart[lane + 1] - my_ya;
      if (my_nrows > 0) {
        const int pky = (int)s_yspan[my_ya - (ya0 & ~3)];
        my_ry0 = pky & 0xffff;
        my_rys = pky >> 16;
      }
      if (warp == 0) {
        Up2Group g;
        g.row = my_ya - ya0;
        g.nrows = my_nrows;
        g.trow = (staged ? my_ry0 - clr0 : my_ry0) * tap_stride;
        g.rys = my_rys;
        s_grp[lane] = g;
      }
    }
    for (int u = warp; u < nw; u += kWarps) {
      const int wi = wA + u;
      const int x0 = min(wi << 5, ow - 1);
      const int x1 = min(x0 + 31, ow - 1);
      const uint32_t valid = (x1 - x0 == 31) ? 0xffffffffu : ((1u << (x1 - x0 + 1)) - 1u);
      const int p0 = (int)s_xspan[x0 - (wA << 5)], p1 = (int)s_xspan[x1 - (wA << 5)];
      const int c0 = p0 & 0xffff;
      const int c1 = (p1 & 0xffff) + (p1 >> 16);  // exclusive
      const int cw0 = c0 >> 5;
      const bool two_words = ((c1 - 1) >> 5) <= cw0 + 1;
      uint32_t m0, m1 = 0;
      {
        const int lo = c0 - (cw0 << 5), hi = min(c1 - (cw0 << 5), 32);
        m0 = (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
        const int hi1 = c1 - ((cw0 + 1) << 5);
        if (hi1 > 0) m1 = hi1 >= 32 ? 0xffffffffu : ((1u << hi1) - 1u);
      }
      // 0 = all background, 1 = all foreground (and safe), 2 = boundary word
      int cls = 0;
      if (my_nrows > 0) {
        const int lrb = (my_ry0 - clr0) * lr_wpr + cw0;
        bool all0 = true, all1 = true;
        if (two_words) {
          uint32_t any = 0, miss = 0;
          for (int r = 0; r < my_rys; ++r) {
            const uint32_t v0 = s_lr[lrb + r * lr_wpr] & m0;
            const uint32_t v1 = s_lr[lrb + r * lr_wpr + 1] & m1;
            any |= v0 | v1;
            miss |= (v0 ^ m0) | (v1 ^ m1);
          }
          all0 = any == 0;
          all1 = miss == 0;
        } else {
          for (int r = 0; r < my_rys; ++r) {
            const uint32_t* row = s_lr + (lrb - cw0) + r * lr_wpr;
            for (int cw = cw0; cw <= (c1 - 1) >> 5; ++cw) {
              const int lo = max(c0 - (cw << 5), 0), hi = min(c1 - (cw << 5), 32);
              const uint32_t m = (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
              const uint32_t v = row[cw] & m;
              all0 = all0 && (v == 0);
              all1 = all1 && (v == m);
            }
          }
        }
        cls = all0 ? 0 : ((all1 && safe) ? 1 : 2);
        if (cls != 2) {
          const uint32_t word = cls == 1 ? valid : 0u;
          const int row = my_ya - ya0;
          for (int j = 0; j < my_nrows; ++j) s_out[u * kUp2OutStride + (row + j) + ((row + j) >> 5)] = word;
        }
      }
      const uint32_t mixed = __ballot_sync(kFull, cls == 2);
      if (lane == 0) s_mix[u] = mixed;
    }
    __syncthreads();
    // ---- the item's boundary words as one list, so that the warps share them evenly whatever their distribution
    int n_list = 0;
    {
      int off = 0;  // every warp computes the (<= 8) offsets; warp w writes the entries of its columns
      for (int u = 0; u < nw; ++u) {
        const uint32_t mixed = s_mix[u];
        if ((u & (kWarps - 1)) == warp && ((mixed >> lane) & 1u))
          s_list[off + __popc(mixed & ((1u << lane) - 1u))] = (uint16_t)((u << 5) | lane);
        off += __popc(mixed);
      }
      n_list = off;
    }
    __syncthreads();
    // ---- phase B: evaluation, lane = pixel of the word
    if (staged)
      up2_evaluate<true>(warp, lane, n_list, s_list, s_grp, s_xspan, s_xw, s_yw + (ya0 & 3), s_out, src, tile_saddr,
                         tap_stride, tap_c0);
    else
      up2_evaluate<false>(warp, lane, n_list, s_list, s_grp, s_xspan, s_xw, s_yw + (ya0 & 3), s_out, src, tile_saddr,
                          tap_stride, tap_c0);
    __syncthreads();
    // ---- epilogue: area and box from the result words, which leave as the word-column-major copy [k][word][row]
    //      (nullable: the overlap windows mask_ios walks are a few words wide and hundreds of rows tall — 4 useful bytes
    //      per 32-byte sector in the row-major layout, contiguous here; the result tile is column-major already, so a
    //      warp writes 128 contiguous bytes per store) and/or row-major in 32-byte row segments
    {
      int area = 0, minx = kBig, maxx = -1, miny = kBig, maxy = -1;
      if (bits_t) {  // warp = word column, lane = row
        uint32_t* dt = bits_t + (size_t)k * oh * ow_words;
        for (int c = warp; c < nw; c += kWarps) {
          uint32_t colbits = 0;
          for (int row = lane; row < n_rows; row += 32) {
            const uint32_t w = s_out[c * kUp2OutStride + row + (row >> 5)];
            dt[(uint32_t)((wA + c) * oh + ya0 + row)] = w;
            area += __popc(w);
            colbits |= w;
            if (w) { miny = min(miny, ya0 + row); maxy = max(maxy, ya0 + row); }
          }
          if (colbits) {
            minx = min(minx, ((wA + c) << 5) + __ffs(colbits) - 1);
            maxx = max(maxx, ((wA + c) << 5) + 31 - __clz(colbits));
          }
        }
      }
      if (bits_full) {  // thread = (row, word column)
        uint32_t* dst = bits_full + (size_t)k * oh * ow_words;
        const int c = tid & (kUp2Cols - 1);
        uint32_t colbits = 0;
        if (c < nw) {
          for (int row = tid >> 3; row < n_rows; row += kUp2Threads / kUp2Cols) {
            const uint32_t w = s_out[c * kUp2OutStride + row + (row >> 5)];
            dst[(uint32_t)((ya0 + row) * ow_words + wA + c)] = w;
            if (!bits_t) {
              area += __popc(w);
              colbits |= w;
              if (w) { miny = min(miny, ya0 + row); maxy = max(maxy, ya0 + row); }
            }
          }
        }
        if (colbits) {
          minx = ((wA + c) << 5) + __ffs(colbits) - 1;
          maxx = ((wA + c) << 5) + 31 - __clz(colbits);
        }
      }
      area = warp_sum(area);
      minx = warp_min(minx); miny = warp_min(miny); maxx = warp_max(maxx); maxy = warp_max(maxy);
      if (lane == 0) {
        atomicAdd(&s_red[0], area);
        atomicMax(&s_red[1], maxx + 1);
        atomicMax(&s_red[2], maxy + 1);
        atomicMax(&s_red[3], kBig - minx);
        atomicMax(&s_red[4], kBig - miny);
      }
    }
    __syncthreads();
    if (tid == 0) {
      pend_k = k;
#pragma unroll
      for (int q = 0; q < 5; ++q) pend[q] = s_red[q];
      s_item = next;
    }
  }
  if (tid == 0 && pend_k >= 0) up2_publish(pend_k, pend, scratch, area_full, box_full);
}

// shared-memory layout of upsample_pack2_kernel in bytes, without / with a logit tile of `tile_floats`
static size_t up2_fixed_smem(int ih, int iw) {
  const size_t lr_words = (((size_t)ih * (iw / 32) + 4) + 3) & ~(size_t)3;
  return (sizeof(float2) + sizeof(uint32_t)) * (kUp2Cols * 32 + kUp2Rows + 4) + sizeof(float2) * 4 +
         sizeof(Up2Group) * kUp2Groups +
         4 * ((size_t)kUp2Cols * kUp2OutStride + kUp2Groups + 4 + lr_words) + 2 * (size_t)kUp2Cols * kUp2Groups;
}
// items a selection can expand to: every mask at most ceil(groups / 32) x ceil(words / 8), groups <= output rows
static size_t up2_max_items(int max_sel, int oh, int ow) {
  return (size_t)max_sel * ((oh + kUp2Groups - 1) / kUp2Groups) * ((((ow + 31) / 32) + kUp2Cols - 1) / kUp2Cols);
}

// one axis's factor of the v2 tile budget: the input rows (columns) an item of kUp2Rows rows (kUp2Cols words) spans at
// this scale, plus slack
long up2_tile_factor(int in_size, int out_size, bool rows) {
  const double sc = (double)in_size / out_size;
  return rows ? (long)((kUp2Rows * sc + 6)) : (long)(((kUp2Cols * 32) * sc + 12));
}

// The full-resolution resize: the general chain (upsample_meta + upsample_pack), the two-tap chain (upsample_plan +
// upsample_pack2) or both.
// Static size (sized == nullptr): the tables tx, ty of oh x ow; the two-tap chain when both axes have two-tap records
// and the size fits its 16-bit item fields and its shared memory, the general chain otherwise.
// Sized entry (sized, atlas; tx, ty are not read): oh x ow is the capacity, which sets the launch shapes and shared
// memory (with the largest tile budget of the range); each kernel reads the size and its tables when it runs.  Sizes of
// the range that take the general path (an axis reaching below the low-res size, see aa_spans_within_two) enqueue its
// chain as well, and the chain the size does not select exits at its first instruction.
// bits_t (nullable): the two-tap chain writes the word-column-major copy [k][word][row] instead of the row-major words
// (every consumer of the fused pipeline reads it) unless a general chain is enqueued as well: the consumers then read
// one layout whichever chain ran.  *wrote_t tells which layout was written; zero2 (nullable: two counters of the next
// stage) is zeroed only when it is the transposed one.
int launch_upsample_pack(const AxisTable& tx, const AxisTable& ty, const float* logits, const uint32_t* bits_lr,
                         const int32_t* box_lr, const int32_t* flags_lr, int ih, int iw, const int32_t* sel,
                         const int32_t* n_sel, int max_sel, int oh, int ow, uint32_t* bits_full, int32_t* rect,
                         int32_t* area_full, int32_t* box_full, int32_t* scratch, const float* const* mask_ptr,
                         cudaStream_t s, int stage_floats, int sm_count, uint32_t* bits_t, bool* wrote_t,
                         bool low_latency, int32_t* zero2, const SizedDims* sized, const SizedAtlas* atlas) {
  if (wrote_t) *wrote_t = false;
  if (max_sel <= 0) return NTTT_OK;
  if (iw % 32 != 0) return NTTT_EUNSUPPORTED;
  const bool two_tap_fits = oh < 65536 && ow < 65536 && ih * (iw / 32) <= 16384;
  bool general, two_tap;
  long budget;  // the two-tap chain's logit tile: what an item of 32 groups x 8 words needs at this scale (+ slack)
  UpTables t{};
  if (sized) {
    general = atlas->any_general;
    two_tap = atlas->any_two_tap;
    if (two_tap && !two_tap_fits) return NTTT_EUNSUPPORTED;
    budget = atlas->max_budget;
  } else {
    two_tap = tx.pk_span && ty.pk_span && two_tap_fits;
    general = !two_tap;
    budget = up2_tile_factor(ih, oh, true) * up2_tile_factor(iw, ow, false);
    t = UpTables{tx.xmin, tx.xsize, tx.w, tx.taps, ty.xmin, ty.xsize, ty.w, ty.taps, tx.t_lo, tx.t_len, ty.t_lo,
                 ty.t_len, ty.grp_of, ty.grp_start, tx.pk_span, tx.pk_w, ty.pk_span, ty.pk_w};
  }
  // general: bits (+ one spare word read and masked off by the footprint test), padded to 16 bytes, then the logit tile
  const size_t bits_bytes = ((((size_t)ih * (iw / 32) + 1) + 3) & ~(size_t)3) * 4;
  if (general && bits_bytes > 160 * 1024) return NTTT_EUNSUPPORTED;
  size_t stage_bytes = (size_t)(stage_floats > 0 ? stage_floats : 0) * 4;
  if (bits_bytes + stage_bytes > 200 * 1024) stage_bytes = 0;
  const size_t smem1 = bits_bytes + stage_bytes;
  // two-tap
  const int tile_floats = up2_tile_floats(budget, stage_floats);
  const size_t smem2 = up2_fixed_smem(ih, iw) + (size_t)tile_floats * 4;
  if (two_tap && smem2 > 200 * 1024) return NTTT_EUNSUPPORTED;
  const bool t_layout = two_tap && !general && bits_t;

  const SizedDims d = sized ? *sized : SizedDims{};
  UpMeta* meta = reinterpret_cast<UpMeta*>(scratch + (size_t)kScratchInts * max_sel);
  if (general) {
    const auto pack = sized ? upsample_pack_kernel<true> : upsample_pack_kernel<false>;
    if (smem1 > 48 * 1024) NTTT_CUDA(set_dyn_smem(pack, (int)smem1));
    (sized ? upsample_meta_kernel<true> : upsample_meta_kernel<false>)<<<ceil_div(max_sel, 256), 256, 0, s>>>(
        bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, t, meta, rect, scratch, logits, mask_ptr, d);
    NTTT_LAUNCH_CHECK();
    pack<<<dim3(kUpMaxSplit, max_sel), kUpThreads, smem1, s>>>(bits_lr, meta, ih, iw, n_sel, max_sel, oh, ow, t,
                                                               bits_full, area_full, box_full, scratch,
                                                               (int)(stage_bytes / 4), d);
    NTTT_LAUNCH_CHECK();
  }
  if (two_tap) {
    int32_t* ctr = reinterpret_cast<int32_t*>(meta + max_sel);
    Up2Item* items = reinterpret_cast<Up2Item*>(ctr + 4);
    // (eight CTAs: the geometry pass is redundant per CTA, the item records are shared out)
    launch_chain(sized ? upsample_plan_kernel<true> : upsample_plan_kernel<false>, 8, kPlanThreads, 0, s, bits_lr,
                 box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, t, meta, rect, scratch, logits, mask_ptr, items, ctr,
                 area_full, box_full, oh, ow, tile_floats, stage_floats, !general, d);
    NTTT_LAUNCH_CHECK();
    const auto pack2 = sized ? upsample_pack2_kernel<true> : upsample_pack2_kernel<false>;
    if (smem2 > 48 * 1024) NTTT_CUDA(set_dyn_smem(pack2, (int)smem2));
    // many images in flight: one persistent CTA per SM leaves the rest of the SM to the other images' kernels (measured
    // 89.8 / 90.7 / 91.2 / 91.9 us/image with 1 / 2 / 3 / 7 CTAs per SM); one image: kUp2CtasPerSm for the shortest kernel
    const int grid = (sm_count > 0 ? sm_count : 148) * (low_latency ? kUp2CtasPerSm : 1);
    launch_chain(pack2, grid, kUp2Threads, smem2, s, bits_lr, meta, ih, iw, oh, ow, t, t_layout ? nullptr : bits_full,
                 t_layout ? bits_t : nullptr, area_full, box_full, scratch, items, ctr, t_layout ? zero2 : nullptr, d);
    NTTT_LAUNCH_CHECK();
  }
  if (wrote_t) *wrote_t = t_layout;
  return NTTT_OK;
}

size_t upsample_scratch_bytes(int max_sel, int oh, int ow) {
  return (sizeof(int32_t) * kScratchInts + sizeof(UpMeta)) * (size_t)max_sel + 16 +
         sizeof(Up2Item) * up2_max_items(max_sel, oh, ow);
}

// ---------------------------------------------------------------------------------------------------
// unpack: packed words -> torch.bool bytes.  `index` (nullable) maps output slot j -> packed mask k.
// HBM-bound: oh*ow bytes written per mask.  One thread expands one 32-pixel word into two 128-bit stores
// (nibble -> 4 bytes is one multiply and one mask); rows outside the mask's rect are zero-filled unread.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t nibble_to_bytes(uint32_t nb) { return (nb * 0x00204081u) & 0x01010101u; }

constexpr int kUnpackRows = 32;   // output rows per CTA
constexpr int kUnpackUnroll = 4;  // words per thread in flight

// (oh, ow): the size of the packed masks; output plane j starts at out + j * oplane, rows are ostride bytes apart and
// bytes up to ostride may be written (the pad bits of the last word are zero).  A static size has ostride = ow,
// oplane = oh * ow; the kSized instance keeps the capacity's strides and writes the [oh, ow] corner of the plane for the
// size read on the device (out of range: the count is zero).
template <bool kSized>
__global__ void __launch_bounds__(256)
unpack_masks_kernel(const uint32_t* __restrict__ bits_full, const int32_t* __restrict__ rect,
                    const int32_t* __restrict__ index, const int32_t* __restrict__ count, int max_count, int oh, int ow,
                    uint8_t* __restrict__ out, bool tr /* packed words are [word][row] instead of [row][word] */,
                    SizedDims d) {
  const int ostride = kSized ? d.cap_w : ow;
  const size_t oplane = kSized ? (size_t)d.cap_h * d.cap_w : (size_t)oh * ow;
  if constexpr (kSized) sized_hw(d, oh, ow);
  const int j = blockIdx.y;
  if (j >= min(*count, max_count)) return;
  const int k = index ? index[j] : j;
  const int ow_words = (ow + 31) >> 5;
  const int4 rc = reinterpret_cast<const int4*>(rect)[k];
  const uint32_t* src = bits_full + (size_t)k * oh * ow_words;
  uint8_t* dst = out + (size_t)j * oplane;
  const int y0 = blockIdx.x * kUnpackRows;
  const int rows = min(kUnpackRows, oh - y0);
  const bool vec = (ostride & 15) == 0;  // every 16-pixel half word starts 16-byte aligned
  const int total = rows * ow_words;
  for (int base = 0; base < total; base += 256 * kUnpackUnroll) {
    uint32_t word[kUnpackUnroll];
    int yy[kUnpackUnroll], ww[kUnpackUnroll];
#pragma unroll
    for (int u = 0; u < kUnpackUnroll; ++u) {  // all loads first
      const int it = base + u * 256 + threadIdx.x;
      const int ry = it / ow_words;
      yy[u] = y0 + ry;
      ww[u] = it - ry * ow_words;
      word[u] = 0;
      if (it < total && yy[u] >= rc.x && yy[u] < rc.y && ww[u] >= rc.z && ww[u] < rc.w)
        word[u] = __ldg(tr ? src + (size_t)ww[u] * oh + yy[u] : src + (size_t)yy[u] * ow_words + ww[u]);
    }
#pragma unroll
    for (int u = 0; u < kUnpackUnroll; ++u) {
      const int it = base + u * 256 + threadIdx.x;
      if (it >= total) continue;
      const int x = ww[u] << 5;
      const uint32_t w = word[u];
      uint8_t* p = dst + (size_t)yy[u] * ostride + x;
      if (vec) {
        *reinterpret_cast<uint4*>(p) = make_uint4(nibble_to_bytes(w & 15u), nibble_to_bytes((w >> 4) & 15u),
                                                   nibble_to_bytes((w >> 8) & 15u), nibble_to_bytes((w >> 12) & 15u));
        if (x + 16 < ostride)
          *reinterpret_cast<uint4*>(p + 16) = make_uint4(nibble_to_bytes((w >> 16) & 15u), nibble_to_bytes((w >> 20) & 15u),
                                                        nibble_to_bytes((w >> 24) & 15u), nibble_to_bytes(w >> 28));
      } else {
        for (int q = 0; q < 32 && x + q < ostride; ++q) p[q] = (w >> q) & 1u;
      }
    }
  }
}

// Sparse unpack into PERSISTENT output buffers: out[j] still holds the mask the previous call wrote there, whose
// rect is remembered in prev_rect[j] (all-zero buffers and rects initially).  Two passes over one index space:
// the OLD rect is cleared where the new rect does not cover it, then the NEW rect is written — so a call touches
// area(old \ new) + area(new) bytes per mask whatever the distance between the two rects (never their common bounding
// box, and never oh*ow: the dense unpack is HBM-write-bound on mostly zeros).  Every slot up to max_count is visited
// so that slots that fall out of use are cleared.
// (oh, ow), ostride, oplane: as in unpack_masks_kernel (out of range: the count is zero and only the previous rects are
// cleared).  The sized entry's rects of earlier, larger images are cleared up to the capacity's row length, so the whole
// buffer stays the dense result embedded top-left with zeros elsewhere.
// (A function of its own: written inside the kernel, these statements compile to different SASS; this is the one
// measured.)
__device__ __forceinline__ void
unpack_sparse_body(const uint32_t* __restrict__ bits_full, const int32_t* __restrict__ rect,
                   const int32_t* __restrict__ index, const int32_t* __restrict__ count, int max_count, int oh, int ow,
                   int ostride, size_t oplane, uint8_t* __restrict__ out, int32_t* __restrict__ prev_rect, bool tr) {
  const int j = blockIdx.y;
  const int ow_words = (ow + 31) >> 5;
  const bool live = j < min(*count, max_count);
  const int k = live ? (index ? index[j] : j) : 0;
  const int4 nr = live ? reinterpret_cast<const int4*>(rect)[k] : make_int4(0, 0, 0, 0);
  const int4 pr = reinterpret_cast<const int4*>(prev_rect)[j];
  const bool has_new = nr.y > nr.x && nr.w > nr.z, has_old = pr.y > pr.x && pr.w > pr.z;
  __syncthreads();  // every thread has read prev_rect[j] before thread 0 overwrites it
  if (blockIdx.x == 0 && threadIdx.x == 0) reinterpret_cast<int4*>(prev_rect)[j] = has_new ? nr : make_int4(0, 0, 0, 0);
  if (!has_new && !has_old) return;
  const int old_w = has_old ? pr.w - pr.z : 0, new_w = has_new ? nr.w - nr.z : 0;
  const int old_h = has_old ? pr.y - pr.x : 0, new_h = has_new ? nr.y - nr.x : 0;
  const int n_old = has_old ? (pr.y - pr.x) * old_w : 0;
  const int total = n_old + (has_new ? (nr.y - nr.x) * new_w : 0);
  const uint32_t* src = bits_full + (size_t)k * oh * ow_words;
  uint8_t* dst = out + (size_t)j * oplane;
  const bool vec = (ostride & 15) == 0;
  for (int it = blockIdx.x * 256 + threadIdx.x; it < total; it += gridDim.x * 256) {
    int y, wi;
    uint32_t w = 0;
    // (transposed source: consecutive threads take consecutive ROWS of one word column, so the reads are contiguous;
    //  a thread writes a whole 32-byte sector either way)
    if (it < n_old) {  // clearing pass: old words the new rect will not rewrite
      if (tr) { const int cw = it / old_h; wi = pr.z + cw; y = pr.x + (it - cw * old_h); }
      else    { const int ry = it / old_w; y = pr.x + ry; wi = pr.z + (it - ry * old_w); }
      if (has_new && y >= nr.x && y < nr.y && wi >= nr.z && wi < nr.w) continue;
    } else {           // writing pass
      const int q = it - n_old;
      if (tr) { const int cw = q / new_h; wi = nr.z + cw; y = nr.x + (q - cw * new_h); }
      else    { const int ry = q / new_w; y = nr.x + ry; wi = nr.z + (q - ry * new_w); }
      w = __ldg(tr ? src + (size_t)wi * oh + y : src + (size_t)y * ow_words + wi);
    }
    const int x = wi << 5;
    uint8_t* p = dst + (size_t)y * ostride + x;
    if (vec) {
      *reinterpret_cast<uint4*>(p) = make_uint4(nibble_to_bytes(w & 15u), nibble_to_bytes((w >> 4) & 15u),
                                                 nibble_to_bytes((w >> 8) & 15u), nibble_to_bytes((w >> 12) & 15u));
      if (x + 16 < ostride)
        *reinterpret_cast<uint4*>(p + 16) = make_uint4(nibble_to_bytes((w >> 16) & 15u), nibble_to_bytes((w >> 20) & 15u),
                                                      nibble_to_bytes((w >> 24) & 15u), nibble_to_bytes(w >> 28));
    } else {
      for (int q = 0; q < 32 && x + q < ostride; ++q) p[q] = (w >> q) & 1u;
    }
  }
}

template <bool kSized>
__global__ void __launch_bounds__(256)
unpack_sparse_kernel(const uint32_t* __restrict__ bits_full, const int32_t* __restrict__ rect,
                     const int32_t* __restrict__ index, const int32_t* __restrict__ count, int max_count, int oh, int ow,
                     uint8_t* __restrict__ out, int32_t* __restrict__ prev_rect, bool tr, SizedDims d) {
  chain_wait();
  const int ostride = kSized ? d.cap_w : ow;
  const size_t oplane = kSized ? (size_t)d.cap_h * d.cap_w : (size_t)oh * ow;
  if constexpr (kSized) sized_hw(d, oh, ow);
  unpack_sparse_body(bits_full, rect, index, count, max_count, oh, ow, ostride, oplane, out, prev_rect, tr);
}

// sized (nullable): the size is read on the device; oh, ow are then the capacity
int launch_unpack_sparse(const uint32_t* bits_full, const int32_t* rect, const int32_t* index, const int32_t* count,
                         int max_count, int oh, int ow, uint8_t* out, int32_t* prev_rect, cudaStream_t s, bool tr,
                         const SizedDims* sized) {
  if (max_count <= 0) return NTTT_OK;
  dim3 grid(1, max_count);  // one CTA per slot: prev_rect[j] is read and rewritten by the same CTA
  launch_chain(sized ? unpack_sparse_kernel<true> : unpack_sparse_kernel<false>, grid, 256, 0, s, bits_full, rect, index,
               count, max_count, oh, ow, out, prev_rect, tr, sized ? *sized : SizedDims{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

int launch_unpack(const uint32_t* bits_full, const int32_t* rect, const int32_t* index, const int32_t* count,
                  int max_count, int oh, int ow, uint8_t* out, cudaStream_t s, bool tr, const SizedDims* sized) {
  if (max_count <= 0) return NTTT_OK;
  dim3 grid(ceil_div(oh, kUnpackRows), max_count);
  (sized ? unpack_masks_kernel<true> : unpack_masks_kernel<false>)<<<grid, 256, 0, s>>>(
      bits_full, rect, index, count, max_count, oh, ow, out, tr, sized ? *sized : SizedDims{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
