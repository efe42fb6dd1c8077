// Pooling contraction, L2 normalisation, prototype preparation, cosine similarity and top-1 label.
//
// Reference: compute_sim_global_avg (matching_baseline_utils.py:869-904) and the top-k section
// (Sam2MatchingBaseline_noAMG.py:602-612).
#include <cuda_bf16.h>

#include "common.cuh"

namespace nttt {

// ---------------------------------------------------------------------------------------------------
// rows: x = sums / max(area,1)  (area==0 -> 1, matching_baseline_utils.py:887-888); x /= max(||x||, 1e-12)
// one warp per row.  nan_empty: the negative-reference variant has NO zero guard (matching_baseline_utils.py:925,
// Sam2MatchingBaseline_noAMG.py:598-600): an empty mask divides 0 by 0 and its whole row is NaN, as in the reference.
// ---------------------------------------------------------------------------------------------------
// kCounted (nttt_match_image_counted, both kernels): n is the capacity and keeps the partials' stride; the rows stop at
// the live count
template <bool kCounted>
__global__ void __launch_bounds__(256)
normalize_rows_kernel(const float* __restrict__ sums, int n_partials, const int32_t* __restrict__ area, int n, int c,
                      float* __restrict__ out, bool nan_empty, LiveCount live) {
  const int row = blockIdx.x * 8 + warp_id();
  if (row >= (kCounted ? live_count(live) : n)) return;
  const int lane = lane_id();
  float denom = 1.0f;
  if (area) { const int a = area[row]; denom = (a == 0 && !nan_empty) ? 1.0f : (float)a; }
  const float* src = sums + (size_t)row * c;
  const size_t pstride = (size_t)n * c;  // split-K partials of the pooling GEMM, added in order
  float* dst = out + (size_t)row * c;
  float ss = 0.0f;
  for (int i = lane; i < c; i += 32) {
    float t = src[i];
    for (int z = 1; z < n_partials; ++z) t += src[z * pstride + i];
    const float v = __fdiv_rn(t, denom);
    dst[i] = v;
    ss = fmaf(v, v, ss);
  }
  ss = warp_sum(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);
  __syncwarp();
  for (int i = lane; i < c; i += 32) dst[i] = __fdiv_rn(dst[i], nrm);
}

// Vector path for encoder widths that are multiples of 128 (384, 768, 1024, 1536): one warp per row keeps the
// whole row in registers (one pass over HBM), and also emits the split-bf16 A operand [hi | hi | lo] of the
// similarity GEMM so no separate conversion pass is needed.
template <int kVec, bool kCounted>  // float4 per lane, c = 128 * kVec
__global__ void __launch_bounds__(256)
normalize_split_kernel(const float* __restrict__ sums, int n_partials, const int32_t* __restrict__ area, int n, int cp,
                       float* __restrict__ out, __nv_bfloat16* __restrict__ split, bool nan_empty,
                       const int32_t* __restrict__ perm, LiveCount live) {
  chain_wait();
  constexpr int c = 128 * kVec;
  const int row = blockIdx.x * 8 + warp_id();
  if (row >= (kCounted ? live_count(live) : n)) return;
  const int lane = lane_id();
  float denom = 1.0f;
  if (area) { const int a = area[row]; denom = (a == 0 && !nan_empty) ? 1.0f : (float)a; }
  // perm (nullable): the pooling GEMM ran on spatially ordered rows; mask `row` sits at sums row perm[row]
  const float4* src = reinterpret_cast<const float4*>(sums + (size_t)(perm ? perm[row] : row) * c);
  float4 v[kVec];
#pragma unroll
  for (int i = 0; i < kVec; ++i) v[i] = src[i * 32 + lane];
  for (int z = 1; z < n_partials; ++z) {  // split-K partials of the pooling GEMM, added in order
    const float4* pz = src + z * ((size_t)n * c / 4);
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      const float4 t = pz[i * 32 + lane];
      v[i].x += t.x; v[i].y += t.y; v[i].z += t.z; v[i].w += t.w;
    }
  }
  float ss = 0.0f;
#pragma unroll
  for (int i = 0; i < kVec; ++i) {
    v[i].x = __fdiv_rn(v[i].x, denom); v[i].y = __fdiv_rn(v[i].y, denom);
    v[i].z = __fdiv_rn(v[i].z, denom); v[i].w = __fdiv_rn(v[i].w, denom);
    ss = fmaf(v[i].x, v[i].x, ss); ss = fmaf(v[i].y, v[i].y, ss);
    ss = fmaf(v[i].z, v[i].z, ss); ss = fmaf(v[i].w, v[i].w, ss);
  }
  ss = warp_sum(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);
  float4* dst = reinterpret_cast<float4*>(out + (size_t)row * c);
  __nv_bfloat16* sp = split ? split + (size_t)row * 3 * cp : nullptr;
#pragma unroll
  for (int i = 0; i < kVec; ++i) {
    float4 o;
    o.x = __fdiv_rn(v[i].x, nrm); o.y = __fdiv_rn(v[i].y, nrm);
    o.z = __fdiv_rn(v[i].z, nrm); o.w = __fdiv_rn(v[i].w, nrm);
    dst[i * 32 + lane] = o;
    if (sp) {
      const float e[4] = {o.x, o.y, o.z, o.w};
      __nv_bfloat16 hi[4], lo[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        hi[k] = __float2bfloat16_rn(e[k]);
        lo[k] = __float2bfloat16_rn(e[k] - __bfloat162float(hi[k]));
      }
      const int col = (i * 32 + lane) * 4;
      const uint2 h2 = make_uint2((uint32_t)__bfloat16_as_ushort(hi[0]) | ((uint32_t)__bfloat16_as_ushort(hi[1]) << 16),
                                  (uint32_t)__bfloat16_as_ushort(hi[2]) | ((uint32_t)__bfloat16_as_ushort(hi[3]) << 16));
      const uint2 l2 = make_uint2((uint32_t)__bfloat16_as_ushort(lo[0]) | ((uint32_t)__bfloat16_as_ushort(lo[1]) << 16),
                                  (uint32_t)__bfloat16_as_ushort(lo[2]) | ((uint32_t)__bfloat16_as_ushort(lo[3]) << 16));
      *reinterpret_cast<uint2*>(sp + col) = h2;
      *reinterpret_cast<uint2*>(sp + cp + col) = h2;
      *reinterpret_cast<uint2*>(sp + 2 * cp + col) = l2;
    }
  }
}

// returns 1 if the fused vector path ran (split written), 0 if the caller must use the generic kernels
// live (nullable, both launchers): n is a counted call's capacity, the rows stop at the live count
template <int kVec>
static void launch_normalize_split_vec(int grid, cudaStream_t s, const float* sums, int n_partials, const int32_t* area,
                                       int n, int cp, float* out, __nv_bfloat16* sp, bool nan_empty, const int32_t* perm,
                                       const LiveCount* live) {
  if (live)
    launch_chain(normalize_split_kernel<kVec, true>, grid, 256, 0, s, sums, n_partials, area, n, cp, out, sp, nan_empty,
                 perm, *live);
  else
    launch_chain(normalize_split_kernel<kVec, false>, grid, 256, 0, s, sums, n_partials, area, n, cp, out, sp, nan_empty,
                 perm, LiveCount{});
}

int launch_normalize_split(const float* sums, int n_partials, const int32_t* area, int n, int c, int cp, float* out,
                           void* split, bool nan_empty, cudaStream_t s, const int32_t* perm, const LiveCount* live) {
  if (n <= 0) return 1;
  if (c % 128 != 0 || cp != c) return 0;
  const int grid = ceil_div(n, 8);
  __nv_bfloat16* sp = static_cast<__nv_bfloat16*>(split);
  switch (c / 128) {
    case 3: launch_normalize_split_vec<3>(grid, s, sums, n_partials, area, n, cp, out, sp, nan_empty, perm, live); break;
    case 6: launch_normalize_split_vec<6>(grid, s, sums, n_partials, area, n, cp, out, sp, nan_empty, perm, live); break;
    case 8: launch_normalize_split_vec<8>(grid, s, sums, n_partials, area, n, cp, out, sp, nan_empty, perm, live); break;
    case 12: launch_normalize_split_vec<12>(grid, s, sums, n_partials, area, n, cp, out, sp, nan_empty, perm, live); break;
    default: return 0;
  }
  ++g_launches;
  if (cudaGetLastError() != cudaSuccess) return 0;
  return 1;
}

int launch_normalize_rows(const float* sums, int n_partials, const int32_t* area, int n, int c, float* out,
                          bool nan_empty, cudaStream_t s, const LiveCount* live) {
  if (n <= 0) return NTTT_OK;
  (live ? normalize_rows_kernel<true> : normalize_rows_kernel<false>)<<<ceil_div(n, 8), 256, 0, s>>>(
      sums, n_partials, area, n, c, out, nan_empty, live ? *live : LiveCount{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// prototypes: mean over ALL `shots` slots (unfilled zeros included), then L2-normalise
// (matching_baseline_utils.py:893-894).  One warp per class.
__global__ void __launch_bounds__(256)
proto_prepare_kernel(const float* __restrict__ ins_avg, int n_cls, int shots, int c, float* __restrict__ proto) {
  const int cls = blockIdx.x * 8 + warp_id();
  if (cls >= n_cls) return;
  const int lane = lane_id();
  const float* src = ins_avg + (size_t)cls * shots * c;
  float* dst = proto + (size_t)cls * c;
  float ss = 0.0f;
  for (int i = lane; i < c; i += 32) {
    float acc = 0.0f;
    for (int l = 0; l < shots; ++l) acc += src[(size_t)l * c + i];
    const float m = __fdiv_rn(acc, (float)shots);
    dst[i] = m;
    ss = fmaf(m, m, ss);
  }
  ss = warp_sum(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);
  __syncwarp();
  for (int i = lane; i < c; i += 32) dst[i] = __fdiv_rn(dst[i], nrm);
}

int launch_proto_prepare(const float* ins_avg, int n_cls, int shots, int c, float* proto, cudaStream_t s) {
  if (n_cls <= 0) return NTTT_OK;
  proto_prepare_kernel<<<ceil_div(n_cls, 8), 256, 0, s>>>(ins_avg, n_cls, shots, c, proto);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// torch.topk / argmax ordering: NaN is larger than every number; among equals (and among NaNs) the lowest index wins
__device__ __forceinline__ bool top1_beats(float v, int i, float best, int arg) {
  const bool vn = v != v, bn = best != best;
  if (vn != bn) return vn;
  if (vn) return i < arg;
  return v > best || (v == best && i < arg);
}
// torch.clamp(min=0) keeps NaN (fmaxf would drop it)
__device__ __forceinline__ float clamp_min0(float x) { return x < 0.0f ? 0.0f : x; }

// top-1 over classes (lowest index on ties == torch.topk/argmax on CPU); when n_cls == 1 the reference's
// `k == n_cls` branch applies: score *= (score > 0.6*score)  (Sam2MatchingBaseline_noAMG.py:606-609).
// `part` holds n_splits split-K partial similarity matrices (stride split_stride floats); they are summed here
// in a fixed order and the sum is written to `sim` (if non-null).
// kBank (nttt_match_image_banked): n_cls is the bank's capacity (the strides stay ld); the arg-max, the `sim` tap and the
// one-class rule take the live class count of *bank.  The loop stops there: a padded column (similarity 0) must not beat
// a row whose live similarities are all negative.
// kCounted (nttt_match_image_counted): n is the candidate capacity; the rows stop at the live count, and with
// live.split_sm the partials are those gemm_tc_kernel<.., true> left at that count: as many as nttt_match_image adds at
// it, live-count * ld floats apart.
template <bool kBank, bool kCounted>
__global__ void __launch_bounds__(256)
top1_kernel(const float* __restrict__ part, int n_splits, size_t split_stride, float* __restrict__ sim, int ld, int n,
            int n_cls, float* __restrict__ top_score, int32_t* __restrict__ top_label,
            const nttt_match_bank* __restrict__ bank, LiveCount live) {
  chain_wait();
  if constexpr (kCounted) {
    n = live_count(live);
    if (live.split_sm > 0) {
      n_splits = split_count(live.split_k, sim_split_want(n, ld, live.split_k, live.split_sm));
      split_stride = (size_t)n * ld;
    }
  }
  if constexpr (kBank) n_cls = bank->n_cls;
  const int row = blockIdx.x * 8 + warp_id();
  if (row >= n) return;
  const int lane = lane_id();
  const float* src = part + (size_t)row * ld;
  float best = -INFINITY;
  int arg = 0x7fffffff;
  for (int i = lane; i < n_cls; i += 32) {
    float v = src[i];
    for (int z = 1; z < n_splits; ++z) v += src[(size_t)z * split_stride + i];
    if (sim) sim[(size_t)row * ld + i] = v;
    if (top1_beats(v, i, best, arg)) { best = v; arg = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(kFull, best, o);
    const int oa = __shfl_xor_sync(kFull, arg, o);
    if (top1_beats(ob, oa, best, arg)) { best = ob; arg = oa; }
  }
  if (lane == 0) {
    if (n_cls == 1) best = best * (float)(best > __fmul_rn(best, 0.6f));
    top_score[row] = best;
    top_label[row] = arg == 0x7fffffff ? 0 : arg;
  }
}

// bank (nullable): the live class count is read from it (n_cls is then the capacity)
// live (nullable): n is a counted call's capacity (top1_kernel<.., true>)
int launch_top1(const float* part, int n_splits, size_t split_stride, float* sim, int ld, int n, int n_cls,
                float* top_score, int32_t* top_label, cudaStream_t s, const nttt_match_bank* bank, const LiveCount* live) {
  if (n <= 0) return NTTT_OK;
  auto kern = live ? (bank ? top1_kernel<true, true> : top1_kernel<false, true>)
                   : (bank ? top1_kernel<true, false> : top1_kernel<false, false>);
  launch_chain(kern, ceil_div(n, 8), 256, 0, s, part, n_splits, split_stride, sim, ld, n, n_cls, top_score, top_label, bank,
               live ? *live : LiveCount{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// Negative-reference scoring (compute_sim_global_avg_with_neg, matching_baseline_utils.py:906-941) + top-1:
//   sim_pos = clamp(obj . proto_pos[c], 0);  sim_neg = max_l clamp(obj . proto_neg[c, l], 0)
//   sim     = sim_pos * exp(-clamp(sim_neg - sim_pos, 0) / sigma)
// Both similarity matrices arrive as split-K partials and are summed here in a fixed order.
// kBank (nttt_match_image_banked): n_cls and l_neg are the capacity and fix the strides of the partials and of `sim`; the
// loops take the live counts of *bank, whose negatives are packed live_cls x live_l (bank_rows) in the GEMM's columns.
// kCounted: as top1_kernel, for both similarity matrices.
template <bool kBank, bool kCounted>
__global__ void __launch_bounds__(256)
neg_top1_kernel(const float* __restrict__ part_pos, int splits_pos, size_t stride_pos,
                const float* __restrict__ part_neg, int splits_neg, size_t stride_neg, int n, int n_cls, int l_neg,
                float sigma, float* __restrict__ sim, float* __restrict__ top_score, int32_t* __restrict__ top_label,
                const nttt_match_bank* __restrict__ bank, LiveCount live) {
  chain_wait();
  if constexpr (kCounted) {
    n = live_count(live);
    if (live.split_sm > 0) {
      splits_pos = split_count(live.split_k, sim_split_want(n, n_cls, live.split_k, live.split_sm));
      splits_neg = split_count(live.split_k, sim_split_want(n, n_cls * l_neg, live.split_k, live.split_sm));
      stride_pos = (size_t)n * n_cls;
      stride_neg = (size_t)n * n_cls * l_neg;
    }
  }
  int live_cls = n_cls, live_l = l_neg;
  if constexpr (kBank) {
    live_cls = bank->n_cls;
    live_l = bank->l_neg;
  }
  const int row = blockIdx.x * 8 + warp_id();
  if (row >= n) return;
  const int lane = lane_id();
  const float* pp = part_pos + (size_t)row * n_cls;
  const float* pn = part_neg + (size_t)row * n_cls * l_neg;
  float best = -INFINITY;
  int arg = 0x7fffffff;
  for (int i = lane; i < live_cls; i += 32) {
    float sp = pp[i];
    for (int z = 1; z < splits_pos; ++z) sp += pp[(size_t)z * stride_pos + i];
    sp = clamp_min0(sp);
    float sn = 0.0f;  // clamp(min=0) before the max: the max of clamped values is >= 0; NaN propagates (torch.max)
    for (int l = 0; l < live_l; ++l) {
      float v = pn[i * live_l + l];
      for (int z = 1; z < splits_neg; ++z) v += pn[(size_t)z * stride_neg + i * live_l + l];
      if (sn == sn && (v != v || v > sn)) sn = v;
    }
    const float v = __fmul_rn(sp, expf(__fdiv_rn(__fmul_rn(-1.0f, clamp_min0(__fsub_rn(sn, sp))), sigma)));
    if (sim) sim[(size_t)row * n_cls + i] = v;
    if (top1_beats(v, i, best, arg)) { best = v; arg = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(kFull, best, o);
    const int oa = __shfl_xor_sync(kFull, arg, o);
    if (top1_beats(ob, oa, best, arg)) { best = ob; arg = oa; }
  }
  if (lane == 0) {
    if (live_cls == 1) best = best * (float)(best > __fmul_rn(best, 0.6f));
    top_score[row] = best;
    top_label[row] = arg == 0x7fffffff ? 0 : arg;
  }
}

int launch_neg_top1(const float* part_pos, int splits_pos, size_t stride_pos, const float* part_neg, int splits_neg,
                    size_t stride_neg, int n, int n_cls, int l_neg, float sigma, float* sim, float* top_score,
                    int32_t* top_label, cudaStream_t s, const nttt_match_bank* bank, const LiveCount* live) {
  if (n <= 0) return NTTT_OK;
  auto kern = live ? (bank ? neg_top1_kernel<true, true> : neg_top1_kernel<false, true>)
                   : (bank ? neg_top1_kernel<true, false> : neg_top1_kernel<false, false>);
  launch_chain(kern, ceil_div(n, 8), 256, 0, s, part_pos, splits_pos, stride_pos, part_neg, splits_neg, stride_neg, n, n_cls,
               l_neg, sigma, sim, top_score, top_label, bank, live ? *live : LiveCount{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
