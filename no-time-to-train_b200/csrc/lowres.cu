// Low-resolution mask pass: threshold + bit-pack + area + box + stability counts (one HBM pass over the
// SAM-2 logits), the antialias weight tables, and the projection of packed masks onto the encoder grid.
//
// Reference: Sam2MatchingBaseline_noAMG.py:548-549 (lr_masks > 0), :551-558 (feature upsample),
// sam2/utils/amg.py:158-178 (stability), :305-348 (boxes).
#include <cuda_bf16.h>
#include <stdlib.h>

#include <algorithm>

#include <chrono>
#include <vector>

#include "common.cuh"

namespace nttt {

// ---------------------------------------------------------------------------------------------------
// K1: lowres_pack — HBM-bound streaming kernel, one CTA per mask.
//   algorithmic bytes per mask: 4*P read (+ P/8 written)
// ---------------------------------------------------------------------------------------------------
constexpr int kPackThreads = 256;                  // consumer threads (8 warps)
constexpr int kPackBlock = kPackThreads + 32;      // + one producer warp
constexpr int kPackStages = 4;
constexpr int kPackStageF4 = 4 * kPackThreads;     // float4 per stage: 4 per consumer thread = 16 KB
constexpr int kPackStageBytes = kPackStageF4 * 16;

__device__ __forceinline__ uint32_t pk_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void pk_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pk_smem_u32(bar)), "r"(count));
}
// (the barrier helpers of the streaming loops take SHARED-SPACE ADDRESSES computed once per kernel: converting the generic
//  pointer on every call was 11 % of the low-res pass's instructions)
__device__ __forceinline__ void pk_mbar_expect_tx(uint32_t bar_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pk_mbar_arrive(uint32_t bar_addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}
// Bounded wait: a lost arrive traps (CUDA error) instead of hanging the GPU.  The try_wait carries a suspend-time hint:
// the warp sleeps in the instruction until the phase completes (or ~4 us pass) instead of coming back after the short
// default limit — the kernel is HBM-bound, its consumer warps wait most of the time, and every spin of the old loop was
// seven issue slots taken from the other kernels on the SM (a third of this kernel's 18 M warp instructions).
__device__ __forceinline__ void pk_mbar_wait(uint32_t bar_addr, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 20); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar_addr), "r"(parity), "r"(4000u)
        : "memory");
    if (done) return;
  }
  __trap();
}
// TMA 1-D bulk copy global -> shared, completion counted on an mbarrier.  The logits are read exactly once per
// image and are far larger than L2 (268 MB vs 126 MB): they are fetched with an evict-first L2 policy so that the
// stream does not push the other kernels' working sets (packed masks, features, tables) out of the cache.
__device__ __forceinline__ uint64_t pk_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void pk_bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar_addr,
                                             uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          pk_smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(bar_addr), "l"(policy)
      : "memory");
}

// One CTA per mask.  A producer warp streams the 256 KB of logits through a 4-stage ring of 16 KB TMA bulk
// copies (48 KB in flight per CTA without holding registers); eight consumer warps read each stage with
// conflict-free 128-bit LDS and do the per-element work.  That work is issue-bound before it is HBM-bound
// (5-10 ALU ops per logit), so the loop carries only what has to be done per element: the sign bit, the
// finite-range check and (only if asked, kStab) the two stability counts.  Area and box are derived afterwards
// from the packed words in shared memory.
template <bool kStab>
__global__ void __launch_bounds__(kPackBlock, 3)
lowres_pack_kernel(const float4* __restrict__ logits, int p4 /* pixels/4 per mask */, int words_per_row,
                   float thr_hi, float thr_lo, uint32_t* __restrict__ bits, int32_t* __restrict__ area,
                   int32_t* __restrict__ box, int32_t* __restrict__ stab, float* __restrict__ stab_score,
                   int32_t* __restrict__ flags, const float* __restrict__ gate, float gate_min,
                   const float* const* __restrict__ mask_ptr) {
  extern __shared__ __align__(128) unsigned char s_raw[];
  if (gate && !(gate[blockIdx.x] > gate_min)) {
    // filtered-out candidate (pred_iou <= iou_thr): its logits are never read; publish an empty mask
    const int nw = p4 >> 3;
    uint4* d4 = reinterpret_cast<uint4*>(bits + (size_t)blockIdx.x * nw);
    for (int i = threadIdx.x; i < (nw >> 2); i += kPackBlock) d4[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
      area[blockIdx.x] = 0;
      if (kStab) { stab[2 * blockIdx.x] = 0; stab[2 * blockIdx.x + 1] = 0; }
      if (kStab && stab_score) stab_score[blockIdx.x] = __fdiv_rn(0.0f, 0.0f);  // 0 / 0 counts -> NaN, as torch
      flags[blockIdx.x] = 1;
      reinterpret_cast<int4*>(box)[blockIdx.x] = make_int4(0, 0, 0, 0);
    }
    return;
  }
  float4* s_stage = reinterpret_cast<float4*>(s_raw);                                        // ring
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(s_raw + (size_t)kPackStages * kPackStageBytes);  // p4/8 words
  __shared__ uint64_t s_full[kPackStages], s_empty[kPackStages];
  const uint32_t full_a = pk_smem_u32(s_full), empty_a = pk_smem_u32(s_empty);
  __shared__ int s_red[8];  // area, hi, lo, unsafe, minx, miny, maxx, maxy
  const int n = blockIdx.x;
  // mask_ptr (nullable): where the decoder left mask n's logits (multimask_select_kernel); else the dense [n,h,w] array
  const float4* src = mask_ptr ? reinterpret_cast<const float4*>(mask_ptr[n]) : logits + (size_t)n * p4;
  const int lane = lane_id(), warp = warp_id();
  const int n_stages = (p4 + kPackStageF4 - 1) / kPackStageF4;
  if (threadIdx.x < 8) s_red[threadIdx.x] = (threadIdx.x == 4 || threadIdx.x == 5) ? 0x7fffffff : (threadIdx.x >= 6 ? -1 : 0);
  if (threadIdx.x == 0) {
    for (int q = 0; q < kPackStages; ++q) { pk_mbar_init(&s_full[q], 1); pk_mbar_init(&s_empty[q], kPackThreads / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  int hi = 0, lo = 0;
  uint32_t unsafe = 0;
  if (warp == kPackThreads / 32) {
    // ===== producer warp =====
    if (lane == 0) {
      const uint64_t l2_policy = pk_policy_evict_first();
      for (int st = 0; st < n_stages; ++st) {
        const int q = st % kPackStages;
        pk_mbar_wait(empty_a + 8u * q, ((st / kPackStages) & 1) ^ 1);
        const int f4 = min(kPackStageF4, p4 - st * kPackStageF4);
        pk_mbar_expect_tx(full_a + 8u * q, (uint32_t)f4 * 16u);
        pk_bulk_load(s_stage + (size_t)q * kPackStageF4, src + (size_t)st * kPackStageF4, (uint32_t)f4 * 16u, full_a + 8u * q, l2_policy);
      }
    }
  } else {
    // ===== consumer warps =====
    // a positive logit is "safe" iff 2^-100 < v < 2^100: bit pattern strictly between 0x0D800000 and 0x71800000
    constexpr uint32_t kLoBits = 0x0D800000u, kSpan = 0x71800000u - 0x0D800001u;
    for (int st = 0; st < n_stages; ++st) {
      const int q = st % kPackStages;
      pk_mbar_wait(full_a + 8u * q, (st / kPackStages) & 1);
      const float4* buf = s_stage + (size_t)q * kPackStageF4;
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)  // (a short last stage leaves the tail of the slot stale: read zeros instead)
        v[u] = (st * kPackStageF4 + u * kPackThreads + (int)threadIdx.x < p4) ? buf[u * kPackThreads + threadIdx.x]
                                                                              : make_float4(0.f, 0.f, 0.f, 0.f);
      __syncwarp();
      if (lane == 0) pk_mbar_arrive(empty_a + 8u * q);  // this warp has copied its share out of the slot
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int qi = st * kPackStageF4 + u * kPackThreads + threadIdx.x;
        const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        uint32_t nib = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const bool pos = e[k] > 0.0f;
          nib |= (uint32_t)pos << k;
          const bool in_range = (__float_as_uint(e[k]) - (kLoBits + 1u)) < kSpan;
          unsafe |= (uint32_t)(pos && !in_range);
          if (kStab) {
            hi += e[k] > thr_hi;
            lo += e[k] > thr_lo;
          }
        }
        uint32_t word = nib << (4 * (lane & 7));
        word |= __shfl_xor_sync(kFull, word, 1);
        word |= __shfl_xor_sync(kFull, word, 2);
        word |= __shfl_xor_sync(kFull, word, 4);
        if ((lane & 7) == 0 && qi < p4) s_bits[qi >> 3] = word;
      }
    }
  }
  __syncthreads();  // s_bits complete
  // area and box from the packed words; 128-bit stores of the words
  const int n_words = p4 >> 3;
  int a = 0, minx = 0x7fffffff, miny = 0x7fffffff, maxx = -1, maxy = -1;
  for (int wi = threadIdx.x; wi < n_words; wi += kPackBlock) {
    const uint32_t word = s_bits[wi];
    if (word) {
      a += __popc(word);
      const int row = wi / words_per_row;
      const int x0 = (wi - row * words_per_row) * 32;
      minx = min(minx, x0 + __ffs(word) - 1);
      maxx = max(maxx, x0 + 31 - __clz(word));
      miny = min(miny, row);
      maxy = max(maxy, row);
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(bits + (size_t)n * n_words);
  const uint4* s4 = reinterpret_cast<const uint4*>(s_bits);
  for (int i = threadIdx.x; i < (n_words >> 2); i += kPackBlock) dst[i] = s4[i];
  a = warp_sum(a);
  unsafe = (uint32_t)warp_max((int)unsafe);
  minx = warp_min(minx); miny = warp_min(miny); maxx = warp_max(maxx); maxy = warp_max(maxy);
  if (kStab) { hi = warp_sum(hi); lo = warp_sum(lo); }
  if (lane == 0) {
    atomicAdd(&s_red[0], a); atomicMax(&s_red[3], (int)unsafe);
    atomicMin(&s_red[4], minx); atomicMin(&s_red[5], miny); atomicMax(&s_red[6], maxx); atomicMax(&s_red[7], maxy);
    if (kStab) { atomicAdd(&s_red[1], hi); atomicAdd(&s_red[2], lo); }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    area[n] = s_red[0];
    if (kStab) { stab[2 * n] = s_red[1]; stab[2 * n + 1] = s_red[2]; }
    // calculate_stability_score (sam2/utils/amg.py:158-178): int32 / int32 is a true division in float32; both
    // counts are <= 65 536 (exact), an empty mask divides 0 by 0 -> NaN
    if (kStab && stab_score) stab_score[n] = __fdiv_rn((float)s_red[1], (float)s_red[2]);
    flags[n] = s_red[3] ? 0 : 1;
    const bool empty = s_red[6] < s_red[4] || s_red[7] < s_red[5];
    int4 b = empty ? make_int4(0, 0, 0, 0) : make_int4(s_red[4], s_red[5], s_red[6], s_red[7]);
    reinterpret_cast<int4*>(box)[n] = b;
  }
}

// ---------------------------------------------------------------------------------------------------
// K1b: the variant the stage launches (no stability counts).  Same ring, same outputs, a third of the instructions.
//
// Per logit the loop above spends ~6 ALU-pipe instructions (compare, select, range test, two ORs).  Here a logit costs
// two: one funnel shift that appends its SIGN bit to a per-thread bit string, and half of a 3-input integer min plus
// half of a 3-input integer max over the raw bit patterns (VIMNMX3).  For every float except +0.0 and a positive NaN,
// `v > 0` is the complement of the sign bit; and the running signed max / unsigned min of the bit patterns are exactly
// the largest and the smallest positive logit seen, which is all the finite-range ("safe") flag needs.  A thread whose
// min/max reveal a +0.0 or a positive NaN switches, for the rest of its mask, to the literal per-element arithmetic of
// the kernel above, so masks, boxes, areas and flags are identical in every case.
//
// The 8 lanes that share a 32-pixel word do not OR-reduce four words with 12 shuffles; they run a 3-step
// reduce-scatter (4 shuffles in total for four words): each step halves the set of words a lane is responsible for
// and doubles the lanes it has merged.  Which float4 a lane reads for its "slot" j is chosen (addresses are computed
// once, all reads stay 128-bit and conflict-free) so that every merge is a byte permute or one LOP3:
//   u* = 2*g2 + g0 is the word lane g = (g2 g1 g0) ends up holding; slot j holds word u = j ^ u*;
//   slots 2,3 go to lane g^4, then slot 1 to lane g^1 (nibble interleave), then the half word to lane g^2;
//   words with odd u are held by odd lanes, whose own nibble is the LOW one of a byte, so for those words lane g reads
//   float4 g^1 of the word instead of g.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pk_exact_negbits(const uint4& v, uint32_t& unsafe) {
  constexpr uint32_t kLoBits = 0x0D800000u, kSpan = 0x71800000u - 0x0D800001u;
  const uint32_t e[4] = {v.x, v.y, v.z, v.w};
  uint32_t nib = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool pos = __uint_as_float(e[k]) > 0.0f;
    nib |= (uint32_t)(!pos) << k;
    unsafe |= (uint32_t)(pos && !((e[k] - (kLoBits + 1u)) < kSpan));
  }
  return nib;
}

__device__ __forceinline__ uint32_t pk_sign_chain(uint32_t acc, const uint4& v) {  // appends w,z,y,x: x lands in bit 0
  acc = __funnelshift_l(v.w, acc, 1);
  acc = __funnelshift_l(v.z, acc, 1);
  acc = __funnelshift_l(v.y, acc, 1);
  acc = __funnelshift_l(v.x, acc, 1);
  return acc;
}

__global__ void __launch_bounds__(kPackBlock, 3)
lowres_pack_fast_kernel(const float4* __restrict__ logits, int p4 /* pixels/4 per mask */, int words_per_row,
                        uint32_t* __restrict__ bits, int32_t* __restrict__ area, int32_t* __restrict__ box,
                        int32_t* __restrict__ flags, const float* __restrict__ gate, float gate_min,
                        const float* const* __restrict__ mask_ptr) {
  chain_wait();
  extern __shared__ __align__(128) unsigned char s_raw[];
  if (gate && !(gate[blockIdx.x] > gate_min)) {
    const int nw = p4 >> 3;
    uint4* d4 = reinterpret_cast<uint4*>(bits + (size_t)blockIdx.x * nw);
    for (int i = threadIdx.x; i < (nw >> 2); i += kPackBlock) d4[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
      area[blockIdx.x] = 0;
      flags[blockIdx.x] = 1;
      reinterpret_cast<int4*>(box)[blockIdx.x] = make_int4(0, 0, 0, 0);
    }
    return;
  }
  uint4* s_stage = reinterpret_cast<uint4*>(s_raw);
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(s_raw + (size_t)kPackStages * kPackStageBytes);
  __shared__ uint64_t s_full[kPackStages], s_empty[kPackStages];
  const uint32_t full_a = pk_smem_u32(s_full), empty_a = pk_smem_u32(s_empty);
  __shared__ int s_red[8];  // area, -, -, unsafe, minx, miny, maxx, maxy
  const int n = blockIdx.x;
  const float4* src = mask_ptr ? reinterpret_cast<const float4*>(mask_ptr[n]) : logits + (size_t)n * p4;
  const int lane = lane_id(), warp = warp_id();
  const int n_stages = (p4 + kPackStageF4 - 1) / kPackStageF4;
  if (threadIdx.x < 8) s_red[threadIdx.x] = (threadIdx.x == 4 || threadIdx.x == 5) ? 0x7fffffff : (threadIdx.x >= 6 ? -1 : 0);
  if (threadIdx.x == 0) {
    for (int q = 0; q < kPackStages; ++q) { pk_mbar_init(&s_full[q], 1); pk_mbar_init(&s_empty[q], kPackThreads / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  uint32_t unsafe = 0;
  if (warp == kPackThreads / 32) {
    if (lane == 0) {
      const uint64_t l2_policy = pk_policy_evict_first();
      for (int st = 0; st < n_stages; ++st) {
        const int q = st % kPackStages;
        pk_mbar_wait(empty_a + 8u * q, ((st / kPackStages) & 1) ^ 1);
        const int f4 = min(kPackStageF4, p4 - st * kPackStageF4);
        pk_mbar_expect_tx(full_a + 8u * q, (uint32_t)f4 * 16u);
        pk_bulk_load(s_stage + (size_t)q * kPackStageF4, src + (size_t)st * kPackStageF4, (uint32_t)f4 * 16u, full_a + 8u * q, l2_policy);
      }
    }
  } else {
    const int g = lane & 7;
    const int ustar = ((g >> 2) << 1) | (g & 1);
    const int grp = threadIdx.x & ~7;  // first float4 of this lane group's word, within one 256-float4 slab
    int off[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int u = j ^ ustar;
      off[j] = u * kPackThreads + grp + (g ^ (u & 1));
    }
    const uint32_t sel_a = (g & 4) ? 0x04u : 0x40u;        // bytes {mine, partner's} ordered by g2
    const uint32_t sel_c = (g & 2) ? 0x1504u : 0x5140u;    // half words interleaved by g1
    const int word_slot = ustar * (kPackThreads / 8) + (threadIdx.x >> 3);
    int mx = (int)0x80000000;      // largest bit pattern as a signed int  = largest positive logit (or +inf / +NaN)
    uint32_t mn = 0xffffffffu;     // smallest bit pattern as an unsigned  = smallest non-negative logit (+0.0 -> 0)
    bool exact = false;
    for (int st = 0; st < n_stages; ++st) {
      const int q = st % kPackStages;
      pk_mbar_wait(full_a + 8u * q, (st / kPackStages) & 1);
      const uint4* buf = s_stage + (size_t)q * kPackStageF4;
      const int f0 = st * kPackStageF4;
      uint4 v[4];
      if (f0 + kPackStageF4 <= p4) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = buf[off[j]];
      } else {  // short last stage: the tail of the slot is stale, read -1.0f (not positive, invisible to min/max)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          v[j] = (f0 + (off[j] & ~7) < p4) ? buf[off[j]] : make_uint4(0xbf800000u, 0xbf800000u, 0xbf800000u, 0xbf800000u);
      }
      __syncwarp();
      if (lane == 0) pk_mbar_arrive(empty_a + 8u * q);
      uint32_t a01 = 0, a23 = 0;  // sign bits: slot 0 in bits 0-3, slot 1 in bits 4-7 (resp. slots 2, 3)
      if (!exact) {
        a01 = pk_sign_chain(pk_sign_chain(0u, v[1]), v[0]);
        a23 = pk_sign_chain(pk_sign_chain(0u, v[3]), v[2]);
        int mx1 = mx;
        uint32_t mn1 = mn;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mx1 = __vimax3_s32(mx1, (int)v[j].x, (int)v[j].y);
          mx1 = __vimax3_s32(mx1, (int)v[j].z, (int)v[j].w);
          mn1 = __vimin3_u32(mn1, v[j].x, v[j].y);
          mn1 = __vimin3_u32(mn1, v[j].z, v[j].w);
        }
        if (mn1 == 0u || mx1 > 0x7f800000) exact = true;  // +0.0 or a positive NaN: sign bit != !(v > 0)
        else { mx = mx1; mn = mn1; }
      }
      if (exact) {
        a01 = pk_exact_negbits(v[0], unsafe) | (pk_exact_negbits(v[1], unsafe) << 4);
        a23 = pk_exact_negbits(v[2], unsafe) | (pk_exact_negbits(v[3], unsafe) << 4);
      }
      const uint32_t r = __shfl_xor_sync(kFull, a23, 4);
      const uint32_t y = __byte_perm(a01, r, sel_a);
      const uint32_t z = __shfl_xor_sync(kFull, y, 1);
      const uint32_t hv = ~((y & 0x0F0Fu) | (z & 0xF0F0u));  // complement: sign bits -> (v > 0) bits
      const uint32_t z2 = __shfl_xor_sync(kFull, hv, 2);
      const uint32_t word = __byte_perm(hv, z2, sel_c);
      if (!(g & 2) && f0 + ustar * kPackThreads + grp < p4) s_bits[st * (kPackStageF4 / 8) + word_slot] = word;
    }
    // positives seen by the sign-bit path: safe iff 2^-100 < v < 2^100 for all of them
    unsafe |= (uint32_t)(mx >= 0x71800000 || mn < 0x0D800001u);
  }
  __syncthreads();
  const int n_words = p4 >> 3;
  int a = 0, minx = 0x7fffffff, miny = 0x7fffffff, maxx = -1, maxy = -1;
  for (int wi = threadIdx.x; wi < n_words; wi += kPackBlock) {
    const uint32_t word = s_bits[wi];
    if (word) {
      a += __popc(word);
      const int row = wi / words_per_row;
      const int x0 = (wi - row * words_per_row) * 32;
      minx = min(minx, x0 + __ffs(word) - 1);
      maxx = max(maxx, x0 + 31 - __clz(word));
      miny = min(miny, row);
      maxy = max(maxy, row);
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(bits + (size_t)n * n_words);
  const uint4* s4 = reinterpret_cast<const uint4*>(s_bits);
  for (int i = threadIdx.x; i < (n_words >> 2); i += kPackBlock) dst[i] = s4[i];
  a = warp_sum(a);
  unsafe = (uint32_t)warp_max((int)unsafe);
  minx = warp_min(minx); miny = warp_min(miny); maxx = warp_max(maxx); maxy = warp_max(maxy);
  if (lane == 0) {
    atomicAdd(&s_red[0], a); atomicMax(&s_red[3], (int)unsafe);
    atomicMin(&s_red[4], minx); atomicMin(&s_red[5], miny); atomicMax(&s_red[6], maxx); atomicMax(&s_red[7], maxy);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    area[n] = s_red[0];
    flags[n] = s_red[3] ? 0 : 1;
    const bool empty = s_red[6] < s_red[4] || s_red[7] < s_red[5];
    int4 b = empty ? make_int4(0, 0, 0, 0) : make_int4(s_red[4], s_red[5], s_red[6], s_red[7]);
    reinterpret_cast<int4*>(box)[n] = b;
  }
}

// K1c: persistent form of K1b — two CTAs per SM with a 3-stage ring each, CTA b takes masks b, b + grid, b + 2*grid, ...
//
// With images in flight the stage is a queue of kernels competing for SMs, and K1b (one CTA per mask, three CTAs per
// SM to keep enough bytes in flight) owns every register and all shared memory of an SM while it runs: the other
// kernels of the other images — which hardly touch HBM — cannot run beside the one kernel that is bound by it
// (tools/ablate.py: the marginal costs of the stages ADD UP, 39 us of HBM time + 76 us of everything else).
// Here two CTAs per SM keep 96 KB of bulk copies in flight (HBM needs ~55 KB per SM), the producer runs ahead into the
// next mask while the consumers finish the current one, and what the CTAs do not occupy of the SM's registers and
// shared memory stays free for the kernels of the other images.
// The packed words are double-buffered so that one consumer barrier per mask is enough; the warp that finishes the
// mask's statistics last combines and publishes them.
// ---------------------------------------------------------------------------------------------------

__device__ __forceinline__ void pk_consumer_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(kPackThreads) : "memory"); }

// (min-blocks 3 only caps the registers at 72 per thread: the grid holds two CTAs per SM, and the registers this
// kernel does not take are what the kernels of the other images run in)
template <int kPersistStages>
__global__ void __launch_bounds__(kPackBlock, 3)
lowres_pack_persistent_kernel(const float4* __restrict__ logits, int n_masks, int p4 /* pixels/4 per mask */,
                              int words_per_row, uint32_t* __restrict__ bits, int32_t* __restrict__ area,
                              int32_t* __restrict__ box, int32_t* __restrict__ flags, const float* __restrict__ gate,
                              float gate_min, const float* const* __restrict__ mask_ptr) {
  extern __shared__ __align__(128) unsigned char s_raw[];
  uint4* s_stage = reinterpret_cast<uint4*>(s_raw);
  const int n_words = p4 >> 3;
  uint32_t* s_bits0 = reinterpret_cast<uint32_t*>(s_raw + (size_t)kPersistStages * kPackStageBytes);  // 2 x n_words
  __shared__ uint64_t s_full[kPersistStages], s_empty[kPersistStages];
  const uint32_t full_a = pk_smem_u32(s_full), empty_a = pk_smem_u32(s_empty);
  __shared__ int s_part[2][kPackThreads / 32][8];  // per warp: area, unsafe, minx, miny, maxx, maxy
  __shared__ int s_done[2];
  const int lane = lane_id(), warp = warp_id();
  const int n_stages = (p4 + kPackStageF4 - 1) / kPackStageF4;
  if (threadIdx.x == 0) {
    for (int q = 0; q < kPersistStages; ++q) { pk_mbar_init(&s_full[q], 1); pk_mbar_init(&s_empty[q], kPackThreads / 32); }
    s_done[0] = 0; s_done[1] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == kPackThreads / 32) {
    // ===== producer warp: streams the stages of all of this CTA's (non-gated) masks back to back =====
    if (lane == 0) {
      const uint64_t l2_policy = pk_policy_evict_first();
      int sg = 0;  // stages issued so far (ring position)
      for (int n = blockIdx.x; n < n_masks; n += gridDim.x) {
        if (gate && !(gate[n] > gate_min)) continue;
        const float4* src = mask_ptr ? reinterpret_cast<const float4*>(mask_ptr[n]) : logits + (size_t)n * p4;
        for (int st = 0; st < n_stages; ++st, ++sg) {
          const int q = sg % kPersistStages;
          pk_mbar_wait(empty_a + 8u * q, ((sg / kPersistStages) & 1) ^ 1);
          const int f4 = min(kPackStageF4, p4 - st * kPackStageF4);
          pk_mbar_expect_tx(full_a + 8u * q, (uint32_t)f4 * 16u);
          pk_bulk_load(s_stage + (size_t)q * kPackStageF4, src + (size_t)st * kPackStageF4, (uint32_t)f4 * 16u, full_a + 8u * q, l2_policy);
        }
      }
    }
    return;
  }

  // ===== consumer warps =====
  const int g = lane & 7;
  const int ustar = ((g >> 2) << 1) | (g & 1);
  const int grp = threadIdx.x & ~7;
  int off[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int u = j ^ ustar;
    off[j] = u * kPackThreads + grp + (g ^ (u & 1));
  }
  const uint32_t sel_a = (g & 4) ? 0x04u : 0x40u;
  const uint32_t sel_c = (g & 2) ? 0x1504u : 0x5140u;
  const int word_slot = ustar * (kPackThreads / 8) + (threadIdx.x >> 3);
  int sg = 0, it = 0;
  for (int n = blockIdx.x; n < n_masks; n += gridDim.x) {
    uint4* dst = reinterpret_cast<uint4*>(bits + (size_t)n * n_words);
    if (gate && !(gate[n] > gate_min)) {  // filtered-out candidate: its logits are never read
      for (int i = threadIdx.x; i < (n_words >> 2); i += kPackThreads) dst[i] = make_uint4(0, 0, 0, 0);
      if (threadIdx.x == 0) {
        area[n] = 0;
        flags[n] = 1;
        reinterpret_cast<int4*>(box)[n] = make_int4(0, 0, 0, 0);
      }
      continue;
    }
    const int buf = it & 1;
    ++it;
    uint32_t* s_bits = s_bits0 + (size_t)buf * n_words;
    uint32_t unsafe = 0;
    int mx = (int)0x80000000;
    uint32_t mn = 0xffffffffu;
    bool exact = false;
    for (int st = 0; st < n_stages; ++st, ++sg) {
      const int q = sg % kPersistStages;
      pk_mbar_wait(full_a + 8u * q, (sg / kPersistStages) & 1);
      const uint4* sbuf = s_stage + (size_t)q * kPackStageF4;
      const int f0 = st * kPackStageF4;
      uint4 v[4];
      if (f0 + kPackStageF4 <= p4) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = sbuf[off[j]];
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          v[j] = (f0 + (off[j] & ~7) < p4) ? sbuf[off[j]] : make_uint4(0xbf800000u, 0xbf800000u, 0xbf800000u, 0xbf800000u);
      }
      __syncwarp();
      if (lane == 0) pk_mbar_arrive(empty_a + 8u * q);
      uint32_t a01 = 0, a23 = 0;
      if (!exact) {
        a01 = pk_sign_chain(pk_sign_chain(0u, v[1]), v[0]);
        a23 = pk_sign_chain(pk_sign_chain(0u, v[3]), v[2]);
        int mx1 = mx;
        uint32_t mn1 = mn;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mx1 = __vimax3_s32(mx1, (int)v[j].x, (int)v[j].y);
          mx1 = __vimax3_s32(mx1, (int)v[j].z, (int)v[j].w);
          mn1 = __vimin3_u32(mn1, v[j].x, v[j].y);
          mn1 = __vimin3_u32(mn1, v[j].z, v[j].w);
        }
        if (mn1 == 0u || mx1 > 0x7f800000) exact = true;
        else { mx = mx1; mn = mn1; }
      }
      if (exact) {
        a01 = pk_exact_negbits(v[0], unsafe) | (pk_exact_negbits(v[1], unsafe) << 4);
        a23 = pk_exact_negbits(v[2], unsafe) | (pk_exact_negbits(v[3], unsafe) << 4);
      }
      const uint32_t r = __shfl_xor_sync(kFull, a23, 4);
      const uint32_t y = __byte_perm(a01, r, sel_a);
      const uint32_t z = __shfl_xor_sync(kFull, y, 1);
      const uint32_t hv = ~((y & 0x0F0Fu) | (z & 0xF0F0u));
      const uint32_t z2 = __shfl_xor_sync(kFull, hv, 2);
      const uint32_t word = __byte_perm(hv, z2, sel_c);
      if (!(g & 2) && f0 + ustar * kPackThreads + grp < p4) s_bits[st * (kPackStageF4 / 8) + word_slot] = word;
    }
    unsafe |= (uint32_t)(mx >= 0x71800000 || mn < 0x0D800001u);
    pk_consumer_barrier();  // the mask's words are complete (and everybody has left the previous use of the other buffer)
    int a = 0, minx = 0x7fffffff, miny = 0x7fffffff, maxx = -1, maxy = -1;
    for (int wi = threadIdx.x; wi < n_words; wi += kPackThreads) {
      const uint32_t word = s_bits[wi];
      if (word) {
        a += __popc(word);
        const int row = wi / words_per_row;
        const int x0 = (wi - row * words_per_row) * 32;
        minx = min(minx, x0 + __ffs(word) - 1);
        maxx = max(maxx, x0 + 31 - __clz(word));
        miny = min(miny, row);
        maxy = max(maxy, row);
      }
    }
    const uint4* s4 = reinterpret_cast<const uint4*>(s_bits);
    for (int i = threadIdx.x; i < (n_words >> 2); i += kPackThreads) dst[i] = s4[i];
    a = warp_sum(a);
    unsafe = (uint32_t)warp_max((int)unsafe);
    minx = warp_min(minx); miny = warp_min(miny); maxx = warp_max(maxx); maxy = warp_max(maxy);
    int last = 0;
    if (lane == 0) {
      int* pw = s_part[buf][warp];
      pw[0] = a; pw[1] = (int)unsafe; pw[2] = minx; pw[3] = miny; pw[4] = maxx; pw[5] = maxy;
      __threadfence_block();
      last = atomicAdd(&s_done[buf], 1) == kPackThreads / 32 - 1;
      if (last) {
        __threadfence_block();
        int ta = 0, tu = 0, tminx = 0x7fffffff, tminy = 0x7fffffff, tmaxx = -1, tmaxy = -1;
#pragma unroll
        for (int w = 0; w < kPackThreads / 32; ++w) {
          const volatile int* q = s_part[buf][w];
          ta += q[0]; tu |= q[1];
          tminx = min(tminx, q[2]); tminy = min(tminy, q[3]); tmaxx = max(tmaxx, q[4]); tmaxy = max(tmaxy, q[5]);
        }
        s_done[buf] = 0;  // (next use of this buffer is two masks away, behind a consumer barrier)
        area[n] = ta;
        flags[n] = tu ? 0 : 1;
        const bool empty = tmaxx < tminx || tmaxy < tminy;
        reinterpret_cast<int4*>(box)[n] = empty ? make_int4(0, 0, 0, 0) : make_int4(tminx, tminy, tmaxx, tmaxy);
      }
    }
  }
}

// SM count of the current device (queried once per device)
static int current_sm_count() {
  static int cache[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && cache[dev] > 0) return cache[dev];
  int count = 148;
  cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, dev);
  if (dev >= 0 && dev < 64) cache[dev] = count;
  return count;
}

// nttt_ctx_tune(NTTT_TUNE_LOWRES_PERSISTENT), process-wide: 1 (default) = lowres_pack_persistent_kernel, two CTAs per SM
// with a 3-stage ring each; 0 = lowres_pack_fast_kernel, one CTA per mask (3 resident per SM), which low-latency mode
// always uses.  The two write the same bits; the switch lets tests compare them.  Shapes measured with 16 images in
// flight (us/image, CTAs per SM x ring stages): one CTA per mask 88.2 | 1x7: 90.6 | 2x4: 87.5 | 2x3: 86.7 | 2x2: 88.2 |
// 3x3: 87.7 | 3x2: 89.5 | 2x5: 87.9 | 4x2: 89.1 — the thinnest shape that still covers the HBM latency wins, because
// what it does not occupy runs the other images' kernels.
int g_pack_persistent = 1;

// stab may be NULL: the stability counts (sam2/utils/amg.py:158-178) are not read on the noAMG path
// gate (nullable): per-mask score; masks with !(gate[n] > gate_min) are skipped and published as empty
// mask_ptr (nullable, device [n]): mask n is read from mask_ptr[n] (16-byte aligned) instead of logits + n*h*w
// stab != NULL takes the literal per-element kernel, which also counts the stability thresholds
int launch_lowres_pack(const float* logits, int n, int h, int w, float thr, float off, uint32_t* bits,
                       int32_t* area, int32_t* box, int32_t* stab, int32_t* flags, const float* gate, float gate_min,
                       const float* const* mask_ptr, cudaStream_t s, float* stab_score) {
  const long p = (long)h * w;
  if (n <= 0) return NTTT_OK;
  if (w % 32 != 0 || p % 128 != 0 || p / 32 * 4 > 32 * 1024) return NTTT_EUNSUPPORTED;
  if (!mask_ptr && (reinterpret_cast<uintptr_t>(logits) & 15) != 0) return NTTT_EINVAL;  // TMA bulk copies need 16-byte alignment
  const size_t smem = (size_t)kPackStages * kPackStageBytes + (size_t)(p / 32) * sizeof(uint32_t);
  const float4* src = reinterpret_cast<const float4*>(logits);
  if (stab) {
    NTTT_CUDA(set_dyn_smem(lowres_pack_kernel<true>, (int)smem));
    lowres_pack_kernel<true><<<n, kPackBlock, smem, s>>>(src, (int)(p / 4), w / 32, thr + off, thr - off, bits, area, box,
                                                        stab, stab_score, flags, gate, gate_min, mask_ptr);
  } else if (g_pack_persistent && !t_low_latency) {
    constexpr int kCtasPerSm = 2, kStages = 3;
    const size_t sm = (size_t)kStages * kPackStageBytes + 2 * (size_t)(p / 32) * sizeof(uint32_t);  // (words double-buffered)
    const int grid = min(n, kCtasPerSm * current_sm_count());
    NTTT_CUDA(set_dyn_smem(lowres_pack_persistent_kernel<kStages>, (int)sm));
    lowres_pack_persistent_kernel<kStages><<<grid, kPackBlock, sm, s>>>(src, n, (int)(p / 4), w / 32, bits, area, box, flags,
                                                                        gate, gate_min, mask_ptr);
  } else {
    NTTT_CUDA(set_dyn_smem(lowres_pack_fast_kernel, (int)smem));
    // (first kernel of the chain, behind the fork event of the low-latency mode: an ordinary launch)
    lowres_pack_fast_kernel<<<n, kPackBlock, smem, s>>>(src, (int)(p / 4), w / 32, bits, area, box, flags, gate, gate_min,
                                                        mask_ptr);
  }
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// ---------------------------------------------------------------------------------------------------
// Candidate selection fused into the stage (SURVEY.md §8f rank 2): the SAM-2 decoder is run on batches of
// `chunk_prompts` point prompts and returns, per batch, m mask planes [chunk_prompts, m, h, w] and m predicted IoUs
// per prompt.  The reference keeps `argmax(ious[:, first:]) + first` per prompt
// (Sam2MatchingBaseline_noAMG.py:295-299, first = 1), gathers that plane, concatenates the batches (:423-425) and
// filters `score > iou_thr` (:428-431): three full copies of the logits.  Here only the ADDRESS of the chosen plane is
// resolved; the logits stay in the tensors the decoder returned and are read once, by lowres_pack / upsample_pack,
// through mask_ptr[].  torch.argmax semantics: the first maximal value wins, NaN counts as maximal.
// ---------------------------------------------------------------------------------------------------
// kBound (nttt_match_image_bound): the IoUs' address is read from *ious_at and the chunk bases from bases[] (both inside
// the nttt_match_inputs struct in device memory, written by nttt_match_bind) instead of ious and the by-value table
template <bool kBound>
__global__ void multimask_select_kernel(const float* __restrict__ ious, int n, int m, int first, ChunkTable chunks,
                                        int chunk_prompts, size_t plane_elems, const float** __restrict__ mask_ptr,
                                        float* __restrict__ score, const float* const* __restrict__ ious_at,
                                        const float* const* __restrict__ bases) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if constexpr (kBound) ious = *ious_at;
  const float* row = ious + (size_t)i * m;
  int best = first;
  float bv = row[first];
  for (int j = first + 1; j < m; ++j) {
    const float v = row[j];
    if (v > bv || (v != v && bv == bv)) { bv = v; best = j; }
  }
  const int ch = i / chunk_prompts;
  const float* base = kBound ? bases[ch] : chunks.base[ch];
  mask_ptr[i] = base + ((size_t)(i - ch * chunk_prompts) * m + best) * plane_elems;
  score[i] = bv;
}

// ious_at (nullable): read the IoUs' address and the chunk bases from device memory (ious and chunks are then ignored)
int launch_multimask_select(const float* ious, int n, int m, int first, const ChunkTable& chunks, int chunk_prompts,
                            size_t plane_elems, const float** mask_ptr, float* score, cudaStream_t s,
                            const float* const* ious_at, const float* const* bases) {
  if (n <= 0) return NTTT_OK;
  (ious_at ? multimask_select_kernel<true> : multimask_select_kernel<false>)<<<ceil_div(n, 256), 256, 0, s>>>(
      ious, n, m, first, chunks, chunk_prompts, plane_elems, mask_ptr, score, ious_at, bases);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// Single-plane inputs of the bound entry: mask i's address and score, in the form the multimask path leaves them, so
// that the low-res pass, the iou_thr gate, NMS and the resize run their mask_ptr / plane_score forms unchanged.
__global__ void __launch_bounds__(256)
plane_resolve_kernel(const nttt_match_inputs* __restrict__ in, int n, size_t plane_elems,
                     const float** __restrict__ mask_ptr, float* __restrict__ score) {
  chain_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  mask_ptr[i] = in->logits + (size_t)i * plane_elems;
  score[i] = in->pred_ious[i];
}

int launch_plane_resolve(const nttt_match_inputs* in, int n, size_t plane_elems, const float** mask_ptr, float* score,
                         cudaStream_t s) {
  if (n <= 0) return NTTT_OK;
  launch_chain(plane_resolve_kernel, dim3(ceil_div(n, 256)), dim3(256), 0, s, in, n, plane_elems, mask_ptr, score);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// nttt_match_bind: the struct travels as the kernel's argument and is stored with static indices (one 8-byte word per
// lane and step), so no host buffer is read when the kernel runs
static_assert(sizeof(nttt_match_inputs) % 8 == 0, "nttt_match_inputs is copied in 8-byte words");
__global__ void __launch_bounds__(32) match_bind_kernel(nttt_match_inputs v, nttt_match_inputs* __restrict__ dst) {
  constexpr int kWords = sizeof(nttt_match_inputs) / 8;
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&v);
  unsigned long long* out = reinterpret_cast<unsigned long long*>(dst);
#pragma unroll
  for (int k = 0; k < kWords; ++k)
    if ((k & 31) == (int)threadIdx.x) out[k] = src[k];
}

int launch_match_bind(const nttt_match_inputs& v, nttt_match_inputs* dst, cudaStream_t s) {
  match_bind_kernel<<<1, 32, 0, s>>>(v, dst);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// ---------------------------------------------------------------------------------------------------
// Antialias weight tables.  Exact fp32 recipe (every operation individually rounded, no contraction):
//   scale = in/out; support = scale>=1 ? scale : 1; invscale = scale>=1 ? float(1.0/double(scale)) : 1
//   center = scale*(i+0.5); xmin = max(int(center-support+0.5),0); xsize = min(int(center+support+0.5),in)-xmin
//   w_j = tri((j + (xmin-center) + 0.5)*invscale); w_j /= sum_j w_j (sequential sum)
// ---------------------------------------------------------------------------------------------------
int aa_max_taps(int in_size, int out_size) {
  const float scale = (float)in_size / (float)out_size;
  const float support = scale >= 1.0f ? scale : 1.0f;
  return (int)ceilf(support) * 2 + 1;
}

__global__ void aa_table_kernel(int in_size, int out_size, int taps, int32_t* xmin, int32_t* xsize, float* w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_size) return;
  const float scale = __fdiv_rn((float)in_size, (float)out_size);
  const float support = scale >= 1.0f ? scale : 1.0f;
  const float invscale = scale >= 1.0f ? (float)(1.0 / (double)scale) : 1.0f;
  const float center = __fmul_rn(scale, __fadd_rn((float)i, 0.5f));
  int lo = (int)__fadd_rn(__fsub_rn(center, support), 0.5f);
  lo = max(lo, 0);
  int hi = (int)__fadd_rn(__fadd_rn(center, support), 0.5f);
  hi = min(hi, in_size);
  const int size = hi - lo;
  const float lo_m_center = __fsub_rn((float)lo, center);
  float total = 0.0f;
  float* wi = w + (size_t)i * taps;
  for (int j = 0; j < size; ++j) {
    float x = __fmul_rn(__fadd_rn(__fadd_rn((float)j, lo_m_center), 0.5f), invscale);
    x = fabsf(x);
    const float v = x < 1.0f ? __fsub_rn(1.0f, x) : 0.0f;
    wi[j] = v;
    total = __fadd_rn(total, v);
  }
  if (total != 0.0f)
    for (int j = 0; j < size; ++j) wi[j] = __fdiv_rn(wi[j], total);
  for (int j = size; j < taps; ++j) wi[j] = 0.0f;
  xmin[i] = lo;
  xsize[i] = size;
}

// transposed view: for input coordinate e, outputs [t_lo, t_lo+t_len) are those whose span contains e
__global__ void aa_transpose_kernel(int in_size, int out_size, int taps, const int32_t* xmin, const int32_t* xsize,
                                    const float* w, int32_t* t_lo, int32_t* t_len, float* t_w, float* t_cum) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= in_size) return;
  int lo = -1, hi = -1;
  for (int x = 0; x < out_size; ++x) {
    if (e >= xmin[x] && e < xmin[x] + xsize[x]) {
      if (lo < 0) lo = x;
      hi = x;
    }
  }
  const int len = lo < 0 ? 0 : hi - lo + 1;  // true length; t_w only holds the first kMaxScatter weights
  t_lo[e] = max(lo, 0);
  t_len[e] = len;
  if (!t_w) return;  // (tables of the sized atlas: no scatter view)
  for (int t = 0; t < kMaxScatter; ++t) {
    const int x = lo + t;
    float v = 0.0f;
    if (lo >= 0 && x <= hi && e >= xmin[x] && e < xmin[x] + xsize[x]) v = w[(size_t)x * taps + (e - xmin[x])];
    t_w[(size_t)e * kMaxScatter + t] = v;
  }
  float c = 0.0f;  // running sums, in the order project_masks_kernel used to accumulate them per CTA
  t_cum[(size_t)e * (kMaxScatter + 1)] = 0.0f;
  for (int t = 0; t < kMaxScatter; ++t) {
    c += t_w[(size_t)e * kMaxScatter + t];
    t_cum[(size_t)e * (kMaxScatter + 1) + t + 1] = c;
  }
}

// runs of output coordinates with identical (xmin, xsize), at most kGrpMax long
__global__ void aa_group_kernel(int out_size, const int32_t* xmin, const int32_t* xsize, int32_t* grp_of,
                                int32_t* grp_start) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int g = -1, run = 0;
  for (int i = 0; i < out_size; ++i) {
    const bool same = i > 0 && xmin[i] == xmin[i - 1] && xsize[i] == xsize[i - 1] && run < kGrpMax;
    if (!same) { ++g; grp_start[g] = i; run = 0; }
    grp_of[i] = g;
    ++run;
  }
  for (int k = g + 1; k <= out_size; ++k) grp_start[k] = out_size;
}

// two-tap records for the resize fast path (see AxisTable::pk_span / pk_w)
__global__ void aa_pack_kernel(int out_size, int out_pad, int taps, const int32_t* xmin, const int32_t* xsize,
                               const float* w, uint32_t* pk_span, float2* pk_w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_pad) return;
  uint32_t span = 0;
  float2 e = make_float2(0.f, 0.f);
  if (i < out_size) {
    const int cs = xsize[i];
    const float* wi = w + (size_t)i * taps;
    span = (uint32_t)xmin[i] | ((uint32_t)cs << 16);
    e.x = cs > 0 ? wi[0] : 0.0f;
    e.y = cs > 1 ? wi[1] : 0.0f;
  }
  pk_span[i] = span;
  pk_w[i] = e;
}

// Whether every span of the axis has xsize <= 2: aa_table_kernel's spans restated on the host, the same fp32 operations
// each rounded (the volatile intermediates keep the compiler from contracting them).  Up-scaling gives
// int(c + 1.5) - int(c - 0.5) = 2 (1 at the borders) as long as both sums are exact; when c + 1 rounds up to the next
// half (3 -> 37, 96 -> 608, 160 -> 736, ...) the span is three samples wide and its third weight is 0, which aten still
// multiplies in (an inf or NaN there turns the sample into NaN).  Such axes keep the general path.
static bool aa_spans_within_two(int in_size, int out_size) {
  if (in_size > out_size) return false;
  const float scale = (float)in_size / (float)out_size;
  for (int i = 0; i < out_size; ++i) {
    volatile float center = scale * ((float)i + 0.5f);
    volatile float a = center - 1.0f, b = center + 1.0f;
    const int lo = std::max((int)(a + 0.5f), 0), hi = std::min((int)(b + 0.5f), in_size);
    if (hi - lo > 2) return false;
  }
  return true;
}

// Byte offsets of a table's arrays inside its slab.  scatter = false leaves out the scatter weights (t_w, t_cum), which
// only the mask projection reads.
struct AxisLayout {
  bool packed;
  size_t o_xmin, o_xsize, o_w, o_tlo, o_tlen, o_tw, o_tcum, o_gof, o_gst, o_pks, o_pkw, bytes;
};
static AxisLayout axis_layout(int in_size, int out_size, bool scatter) {
  AxisLayout L{};
  L.packed = in_size < 65536 && aa_spans_within_two(in_size, out_size);
  const int taps = aa_max_taps(in_size, out_size);
  const int out_pad = (out_size + 31) / 32 * 32;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
  L.o_xmin = take(sizeof(int32_t) * out_size);
  L.o_xsize = take(sizeof(int32_t) * out_size);
  L.o_w = take(sizeof(float) * (size_t)out_size * taps);
  L.o_tlo = take(sizeof(int32_t) * in_size);
  L.o_tlen = take(sizeof(int32_t) * in_size);
  L.o_tw = scatter ? take(sizeof(float) * (size_t)in_size * kMaxScatter) : 0;
  L.o_tcum = scatter ? take(sizeof(float) * (size_t)in_size * (kMaxScatter + 1)) : 0;
  L.o_gof = take(sizeof(int32_t) * out_size);
  L.o_gst = take(sizeof(int32_t) * ((size_t)out_size + 1));
  L.o_pks = L.packed ? take(sizeof(uint32_t) * (size_t)out_pad) : 0;
  L.o_pkw = L.packed ? take(sizeof(float2) * (size_t)out_pad) : 0;
  L.bytes = off;
  return L;
}

// builds the table into `slab` (L.bytes, laid out by axis_layout), stream-ordered
static int fill_axis_table(AxisTable& t, int in_size, int out_size, const AxisLayout& L, bool scatter, char* slab,
                           cudaStream_t s) {
  const int out_pad = (out_size + 31) / 32 * 32;
  t.xmin = reinterpret_cast<int32_t*>(slab + L.o_xmin);
  t.xsize = reinterpret_cast<int32_t*>(slab + L.o_xsize);
  t.w = reinterpret_cast<float*>(slab + L.o_w);
  t.t_lo = reinterpret_cast<int32_t*>(slab + L.o_tlo);
  t.t_len = reinterpret_cast<int32_t*>(slab + L.o_tlen);
  t.t_w = scatter ? reinterpret_cast<float*>(slab + L.o_tw) : nullptr;
  t.t_cum = scatter ? reinterpret_cast<float*>(slab + L.o_tcum) : nullptr;
  t.grp_of = reinterpret_cast<int32_t*>(slab + L.o_gof);
  t.grp_start = reinterpret_cast<int32_t*>(slab + L.o_gst);
  t.pk_span = L.packed ? reinterpret_cast<uint32_t*>(slab + L.o_pks) : nullptr;
  t.pk_w = L.packed ? reinterpret_cast<float2*>(slab + L.o_pkw) : nullptr;
  aa_table_kernel<<<ceil_div(out_size, 128), 128, 0, s>>>(in_size, out_size, t.taps, t.xmin, t.xsize, t.w);
  NTTT_LAUNCH_CHECK();
  aa_transpose_kernel<<<ceil_div(in_size, 128), 128, 0, s>>>(in_size, out_size, t.taps, t.xmin, t.xsize, t.w, t.t_lo,
                                                            t.t_len, t.t_w, t.t_cum);
  NTTT_LAUNCH_CHECK();
  aa_group_kernel<<<1, 32, 0, s>>>(out_size, t.xmin, t.xsize, t.grp_of, t.grp_start);
  NTTT_LAUNCH_CHECK();
  if (L.packed) {
    aa_pack_kernel<<<ceil_div(out_pad, 128), 128, 0, s>>>(out_size, out_pad, t.taps, t.xmin, t.xsize, t.w, t.pk_span,
                                                             t.pk_w);
    NTTT_LAUNCH_CHECK();
  }
  return NTTT_OK;
}

// All arrays of a table live in ONE device allocation (`slab`): a table costs one cudaMalloc when a new (in, out) pair is
// first seen and one cudaFree when it is retired, instead of ten of each.
int build_axis_table(AxisTable& t, int in_size, int out_size, cudaStream_t s) {
  t.in_size = in_size;
  t.out_size = out_size;
  t.taps = aa_max_taps(in_size, out_size);
  const AxisLayout L = axis_layout(in_size, out_size, true);
  char* slab = nullptr;
  NTTT_CUDA(cudaMalloc(&slab, L.bytes));
  t.slab = slab;
  return fill_axis_table(t, in_size, out_size, L, true, slab, s);
}

// The atlas of the sized entry: the tables of every output height in [min_h, cap_h] from lr_h and of every width in
// [min_w, cap_w] from lr_w, in one slab with the device index behind them, built with the same kernels as the tables
// of the static entry (so a size's tables are bit for bit the ones nttt_match_image uses) behind ONE synchronisation.
int build_sized_atlas(SizedAtlas& a, cudaStream_t s) {
  const auto t0 = std::chrono::steady_clock::now();
  const int ny = a.cap_h - a.min_h + 1, nx = a.cap_w - a.min_w + 1;
  std::vector<AxisLayout> lay(ny + nx);
  std::vector<size_t> at(ny + nx);
  size_t off = 0;
  for (int i = 0; i < ny + nx; ++i) {
    const bool y = i < ny;
    lay[i] = axis_layout(y ? a.lr_h : a.lr_w, y ? a.min_h + i : a.min_w + (i - ny), false);
    at[i] = off;
    off = align_up(off + lay[i].bytes, 256);
  }
  const size_t o_index = off;
  off = align_up(off + sizeof(SizedAxis) * (ny + nx), 256);
  char* slab = nullptr;
  NTTT_CUDA(cudaMalloc(&slab, off));
  std::vector<SizedAxis> index(ny + nx);
  bool y_packed = false, x_packed = false, y_general = false, x_general = false;
  long y_budget = 0, x_budget = 0;
  for (int i = 0; i < ny + nx; ++i) {
    const bool y = i < ny;
    const int in_size = y ? a.lr_h : a.lr_w, out_size = y ? a.min_h + i : a.min_w + (i - ny);
    AxisTable t{};
    t.in_size = in_size;
    t.out_size = out_size;
    t.taps = aa_max_taps(in_size, out_size);
    const int err = fill_axis_table(t, in_size, out_size, lay[i], false, slab + at[i], s);
    if (err) { cudaStreamSynchronize(s); cudaFree(slab); return err; }
    const long budget = up2_tile_factor(in_size, out_size, y);
    index[i] = SizedAxis{t.xmin, t.xsize, t.w, t.t_lo, t.t_len, t.grp_of, t.grp_start, t.pk_span, t.pk_w, t.taps,
                         (int)budget};
    (y ? y_packed : x_packed) |= lay[i].packed;
    (y ? y_general : x_general) |= !lay[i].packed;
    long& mb = y ? y_budget : x_budget;
    if (budget > mb) mb = budget;
  }
  cudaError_t e = cudaMemcpyAsync(slab + o_index, index.data(), sizeof(SizedAxis) * index.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // (also keeps `index` alive until the copy has run)
  if (e != cudaSuccess) { cudaFree(slab); return cuda_fail(e, "sized atlas build"); }
  a.slab = slab;
  a.bytes = off;
  a.ay = reinterpret_cast<SizedAxis*>(slab + o_index);
  a.ax = a.ay + ny;
  a.any_two_tap = y_packed && x_packed;
  a.any_general = y_general || x_general;
  a.max_budget = y_budget * x_budget;
  a.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return NTTT_OK;
}

void free_axis_table(AxisTable& t) {
  if (t.slab) cudaFree(t.slab);
  t = AxisTable{};
}

// ---------------------------------------------------------------------------------------------------
// K2: project_masks — proj[n, ey, ex] = sum_{y,x} Uy[y,ey] * bit(y,x) * Ux[x,ex]
// (Uy, Ux = antialias upsample matrices encoder grid -> mask grid).  With it
//   masks @ upsample(feat)  ==  proj @ feat           (linearity + separability of the resize)
// so the 2*N*P*C contraction of the reference collapses to 2*N*E*C.  Reads only the packed bits
// (P/8 bytes per mask, L2 resident); compute-bound on the set-bit walk.
// ---------------------------------------------------------------------------------------------------
constexpr int kProjThreads = 256;

struct ProjTables {
  const int32_t* x_lo; const int32_t* x_len; const float* x_cum;  // running sums of the column weights
  const int32_t* y_lo; const int32_t* y_len; const float* y_w;
};

__device__ __forceinline__ void split_bf16_pair(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// One CTA per mask.  Work is confined to the mask's low-res box: rows [top,bottom] for the horizontal pass and
// the encoder cells whose spans touch the box for the vertical pass; everything else is written as zero.
// The horizontal pass walks RUNS of set bits (masks are blobs: one or two runs per row) against prefix sums of
// the weights, one warp per row and one lane per encoder column, so there is no per-bit loop and no division.
// The box is processed in chunks of kProjRows mask rows: the packed rows and the horizontal-pass values of one chunk
// live in shared memory, the vertical pass adds the chunk's rows to per-cell accumulators (shared memory, one owner
// thread per cell, same fma order as a single pass) — 18 KB per CTA instead of 47 KB sized for a full-height box,
// i.e. 8 instead of 4 resident CTAs per SM for a kernel that is a chain of short dependent phases.
// kSplit=false: proj f32 [n, stride];  kSplit=true: bf16 [n, 3*kp] laid out [hi | hi | lo] (the A operand of
// the tcgen05 pooling GEMM), zero padded to kp.
constexpr int kCum = kMaxScatter + 1;
constexpr int kProjRows = 64;

// first and last index e in [0, n) with flag(e) true, evaluated by one warp (n <= 64); returns lo > hi if none
template <typename F>
__device__ __forceinline__ void warp_range(int n, F flag, int& lo, int& hi) {
  const int lane = lane_id();
  const uint32_t b0 = __ballot_sync(kFull, lane < n && flag(lane));
  const uint32_t b1 = __ballot_sync(kFull, lane + 32 < n && flag(lane + 32));
  lo = b0 ? __ffs(b0) - 1 : (b1 ? 32 + __ffs(b1) - 1 : 1);
  hi = b1 ? 63 - __clz(b1) : (b0 ? 31 - __clz(b0) : 0);
}

template <bool kSplit>
__global__ void __launch_bounds__(kProjThreads)
project_masks_kernel(const uint32_t* __restrict__ bits, const int32_t* __restrict__ box, int n_masks, int h,
                     int words_per_row, int eh, int ew, ProjTables t, void* __restrict__ out, int stride_or_kp,
                     const int32_t* __restrict__ perm, uint32_t* __restrict__ active) {
  chain_wait();
  extern __shared__ uint32_t smem[];
  // layout: x_lo[ew] x_len[ew] y_lo[eh] y_len[eh] | bits[rc*wpr] | row[rc*ew] | acc[eh*ew]     (rc = min(h, kProjRows))
  // (the weight tables — running column sums, row weights — are the same for every mask and are read through L1
  // from the prebuilt global tables)
  const int rc = min(h, kProjRows);
  int* s_xlo = reinterpret_cast<int*>(smem);
  int* s_xlen = s_xlo + ew;
  int* s_ylo = s_xlen + ew;
  int* s_ylen = s_ylo + eh;
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(s_ylen + eh);
  float* s_row = reinterpret_cast<float*>(s_bits + rc * words_per_row);
  float* s_acc = s_row + rc * ew;
  const int lane = lane_id(), warp = warp_id();
  constexpr int kWarps = kProjThreads / 32;
  if (eh > 64 || ew > 64) return;  // (checked by the launcher)
  // the span tables are the same for every mask: staged once per CTA, which then walks masks blockIdx.x, +gridDim.x, ...
  for (int i = threadIdx.x; i < ew; i += kProjThreads) { s_xlo[i] = t.x_lo[i]; s_xlen[i] = min(t.x_len[i], kMaxScatter); }
  for (int i = threadIdx.x; i < eh; i += kProjThreads) { s_ylo[i] = t.y_lo[i]; s_ylen[i] = min(t.y_len[i], kMaxScatter); }
  for (int n = blockIdx.x; n < n_masks; n += gridDim.x) {
  __syncthreads();  // tables staged / the previous mask's accumulators and rows are no longer read
  const int4 b = reinterpret_cast<const int4*>(box)[n];
  const uint32_t* src = bits + (size_t)n * h * words_per_row;
  const bool empty = (b.x | b.y | b.z | b.w) == 0 && (src[0] & 1u) == 0;
  // perm (nullable): output row of mask n (the pooling GEMM then runs on spatially ordered rows, see pool_order_kernel);
  // active (nullable): per OUTPUT row, the 64-wide k-blocks of the operand that hold anything but zeros
  const int orow = perm ? perm[n] : n;
  const int top = b.y, bottom = b.w, left = b.x, right = b.z;

  // zero the whole output row first (128-bit stores); the cells the box reaches are overwritten below
  {
    const size_t row_bytes = kSplit ? (size_t)3 * stride_or_kp * 2 : (size_t)stride_or_kp * 4;
    char* o = static_cast<char*>(out) + (size_t)orow * row_bytes;
    if ((row_bytes & 15) == 0) {
      for (int i = threadIdx.x; i < (int)(row_bytes >> 4); i += kProjThreads)
        reinterpret_cast<uint4*>(o)[i] = make_uint4(0, 0, 0, 0);
    } else {
      for (int i = threadIdx.x; i < (int)(row_bytes >> 2); i += kProjThreads) reinterpret_cast<uint32_t*>(o)[i] = 0;
    }
  }
  if (empty) {  // (CTA-uniform)
    if (active && threadIdx.x == 0) active[orow] = 0u;
    continue;
  }
  const int nrows = bottom - top + 1;
  // encoder cells whose spans touch the box
  int ex_lo, ex_hi, ey_lo, ey_hi;
  warp_range(ew, [&](int e) { return s_xlo[e] <= right && s_xlo[e] + s_xlen[e] > left; }, ex_lo, ex_hi);
  warp_range(eh, [&](int e) { return s_ylo[e] <= bottom && s_ylo[e] + s_ylen[e] > top; }, ey_lo, ey_hi);
  const int nex = ex_hi - ex_lo + 1;
  if (nex <= 0 || ey_hi < ey_lo) {  // (CTA-uniform)
    if (active && threadIdx.x == 0) active[orow] = 0u;
    continue;
  }
  if (active && warp == 0) {  // k-blocks touched by the cells [ey_lo, ey_hi] x [ex_lo, ex_hi] (cell index ey * ew + ex)
    uint32_t m = 0;
    if (eh * ew > 32 * 64) {
      m = 0xffffffffu;  // more k-blocks than bits: everything counts as active
    } else {
      for (int ey = ey_lo + lane; ey <= ey_hi; ey += 32) {
        const int k0 = (ey * ew + ex_lo) >> 6, k1 = (ey * ew + ex_hi) >> 6;
        m |= (k1 - k0 >= 31 ? 0xffffffffu : ((2u << (k1 - k0)) - 1u)) << k0;
      }
    }
    m = __reduce_or_sync(kFull, m);
    if (lane == 0) active[orow] = m;
  }
  // every cell (ey, ex) has ONE owner thread for the whole kernel: warp = (ey - ey_lo) % kWarps, lane = (ex - ex_lo) % 32
  for (int ey = ey_lo + warp; ey <= ey_hi; ey += kWarps)
    for (int ex = ex_lo + lane; ex <= ex_hi; ex += 32) s_acc[ey * ew + ex] = 0.0f;

  for (int cb = 0; cb < nrows; cb += rc) {
    const int rows_c = min(rc, nrows - cb);
    const int ctop = top + cb;  // first mask row of this chunk
    if (cb > 0) __syncthreads();  // the previous chunk's rows are no longer read
    for (int i = threadIdx.x; i < rows_c * words_per_row; i += kProjThreads) s_bits[i] = src[ctop * words_per_row + i];
    __syncthreads();
    // horizontal pass: s_row[yy, ex - ex_lo] = sum_x bit(ctop + yy, x) * Ux[x, ex], one warp per row
    for (int yy = warp; yy < rows_c; yy += kWarps) {
      const uint32_t* row = s_bits + yy * words_per_row;
      for (int ex = ex_lo + lane; ex <= ex_hi; ex += 32) {
        const int lo = s_xlo[ex], len = s_xlen[ex];
        const int w0 = lo >> 5, sh = lo & 31;
        const uint32_t wa = row[w0];
        const uint32_t wb = (w0 + 1 < words_per_row) ? row[w0 + 1] : 0u;
        uint32_t f = __funnelshift_r(wa, wb, sh);
        f &= (len >= 32) ? 0xffffffffu : ((1u << len) - 1u);
        const float* cw = t.x_cum + ex * kCum;
        float acc = 0.0f;
        while (f) {  // one iteration per run of set bits
          const int a = __ffs(f) - 1;
          const uint32_t g = ~(f >> a);
          const int run = g ? __ffs(g) - 1 : 32 - a;
          acc += __ldg(cw + a + run) - __ldg(cw + a);
          f = (a + run >= 32) ? 0u : (f >> (a + run)) << (a + run);
        }
        s_row[yy * nex + (ex - ex_lo)] = acc;
      }
    }
    __syncthreads();
    // vertical pass: the chunk's rows are added to the cells they reach (taps in ascending order, as in one pass)
    for (int ey = ey_lo + warp; ey <= ey_hi; ey += kWarps) {
      const int lo = s_ylo[ey], len = s_ylen[ey];
      const float* wv = t.y_w + ey * kMaxScatter;
      const int ta = max(max(top - lo, 0), ctop - lo), tb = min(min(bottom - lo + 1, len), ctop + rows_c - lo);
      if (ta >= tb) continue;  // (warp-uniform)
      for (int ex = ex_lo + lane; ex <= ex_hi; ex += 32) {
        float acc = s_acc[ey * ew + ex];
        for (int q = ta; q < tb; ++q) acc = fmaf(__ldg(wv + q), s_row[(lo + q - ctop) * nex + (ex - ex_lo)], acc);
        s_acc[ey * ew + ex] = acc;
      }
    }
  }
  // output (each thread reads back the cells it owns)
  for (int ey = ey_lo + warp; ey <= ey_hi; ey += kWarps) {
    for (int ex = ex_lo + lane; ex <= ex_hi; ex += 32) {
      const float acc = s_acc[ey * ew + ex];
      const int item = ey * ew + ex;
      if (kSplit) {
        __nv_bfloat16 hi, lo16;
        split_bf16_pair(acc, hi, lo16);
        __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out) + (size_t)orow * 3 * stride_or_kp;
        o[item] = hi;
        o[stride_or_kp + item] = hi;
        o[2 * stride_or_kp + item] = lo16;
      } else {
        static_cast<float*>(out)[(size_t)orow * stride_or_kp + item] = acc;
      }
    }
  }
  }  // masks of this CTA
}

static size_t project_smem_bytes(int h, int w, int eh, int ew) {
  const int rc = h < kProjRows ? h : kProjRows;
  return sizeof(int) * 2 * (size_t)(ew + eh) + sizeof(uint32_t) * (size_t)rc * (w / 32) +
         sizeof(float) * (size_t)rc * ew + sizeof(float) * (size_t)eh * ew;
}

// split=false: out = float [n, out_stride];  split=true: out = bf16 [n, 3*out_stride] with out_stride = kp
int launch_project_masks(const AxisTable& tx, const AxisTable& ty, const uint32_t* bits, const int32_t* box, int n,
                         int h, int w, int eh, int ew, void* out, int out_stride, bool split, cudaStream_t s,
                         const int32_t* perm, uint32_t* active) {
  if (n <= 0) return NTTT_OK;
  if (w % 32 != 0 || eh > 64 || ew > 64) return NTTT_EUNSUPPORTED;
  const size_t smem = project_smem_bytes(h, w, eh, ew);
  if (smem > 200 * 1024) return NTTT_EUNSUPPORTED;
  ProjTables t{tx.t_lo, tx.t_len, tx.t_cum, ty.t_lo, ty.t_len, ty.t_w};
  // throughput mode: two persistent CTAs per SM walk the masks (measured 88.1 vs 89.4 us/image with one CTA per mask:
  // the span tables are staged once per CTA and 1024 CTA launches become 296); low-latency mode: one CTA per mask
  const int grid = t_low_latency ? n : min(n, 2 * current_sm_count());
  if (split) {
    if (smem > 48 * 1024)
      NTTT_CUDA(set_dyn_smem(project_masks_kernel<true>, (int)smem));
    launch_chain(project_masks_kernel<true>, grid, kProjThreads, smem, s, bits, box, n, h, w / 32, eh, ew, t, out, out_stride, perm,
                 active);
  } else {
    if (smem > 48 * 1024)
      NTTT_CUDA(set_dyn_smem(project_masks_kernel<false>, (int)smem));
    project_masks_kernel<false><<<grid, kProjThreads, smem, s>>>(bits, box, n, h, w / 32, eh, ew, t, out, out_stride, perm, active);
  }
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// ---------------------------------------------------------------------------------------------------
// Spatial order of the masks for the pooling GEMM.  A projected mask touches only the encoder cells around its box —
// a quarter of the operand's 64-wide k-blocks on average — but a 128-row tile of masks in arbitrary order touches all
// of them.  Rows ordered along a Z-curve over (top edge, bottom edge) of the low-res box make the union of a tile ~55 % of the k-blocks,
// and gemm_tc_kernel skips the rest (zeros times anything finite).  One CTA: counting sort over the 4096 Morton codes of
// (top >> 2, bottom >> 2); ranks inside a bin are handed out by an atomic, so the order inside a bin is arbitrary — the
// row a mask lands in changes nothing in its result.  perm[n] = row of mask n.
// ---------------------------------------------------------------------------------------------------
constexpr int kOrderBins = 64 * 64;
__global__ void __launch_bounds__(1024)
pool_order_kernel(const int32_t* __restrict__ box, int n, int h, int32_t* __restrict__ perm) {
  chain_wait();
  __shared__ int s_hist[kOrderBins];
  __shared__ int s_warp[33];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kOrderBins; i += 1024) s_hist[i] = 0;
  __syncthreads();
  const int shift = 32 - __clz((h - 1) >> 6);  // rows -> at most 64 bins (h = 256: >> 2)
  constexpr int kMaxPer = 8;  // n <= 8192
  int key[kMaxPer], rank[kMaxPer];
#pragma unroll
  for (int q = 0; q < kMaxPer; ++q) {
    const int i = q * 1024 + tid;
    key[q] = -1;
    if (i < n) {
      const int4 b = reinterpret_cast<const int4*>(box)[i];
      // Morton code of (top, bottom): masks that agree in BOTH edges become neighbours (ordering by one edge first leaves
      // the other spread over a tile; simulated union of a 128-row tile: 56 % vs 58 % at 1024 masks, 42 % vs 51 % at 4096)
      const uint32_t t0 = (uint32_t)min(b.y >> shift, 63), t1 = (uint32_t)min(b.w >> shift, 63);
      uint32_t code = 0;
#pragma unroll
      for (int bit = 0; bit < 6; ++bit) code |= (((t0 >> bit) & 1u) << (2 * bit + 1)) | (((t1 >> bit) & 1u) << (2 * bit));
      key[q] = (int)code;
      rank[q] = atomicAdd(&s_hist[key[q]], 1);
    }
  }
  __syncthreads();
  // exclusive scan of the 4096 bins: four consecutive bins per thread
  int c0 = s_hist[4 * tid], c1 = s_hist[4 * tid + 1], c2 = s_hist[4 * tid + 2], c3 = s_hist[4 * tid + 3];
  const int mine = c0 + c1 + c2 + c3;
  int inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int up = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += up;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = s_warp[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += up;
    }
    s_warp[lane] = winc - w;
  }
  __syncthreads();
  const int base = s_warp[warp] + inc - mine;
  s_hist[4 * tid] = base;
  s_hist[4 * tid + 1] = base + c0;
  s_hist[4 * tid + 2] = base + c0 + c1;
  s_hist[4 * tid + 3] = base + c0 + c1 + c2;
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kMaxPer; ++q) {
    const int i = q * 1024 + tid;
    if (i < n) perm[i] = s_hist[key[q]] + rank[q];
  }
}

int launch_pool_order(const int32_t* box, int n, int h, int32_t* perm, cudaStream_t s) {
  if (n <= 0) return NTTT_OK;
  if (n > 8192) return NTTT_EUNSUPPORTED;
  launch_chain(pool_order_kernel, 1, 1024, 0, s, box, n, h, perm);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
