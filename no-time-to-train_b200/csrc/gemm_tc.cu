// tcgen05 / TMEM / TMA GEMM for the two contractions of the matching stage:
//   pooling     sums[N, C]     = proj[N, E]      * feat[E, C]            (matching_baseline_utils.py:890)
//   similarity  sim [N, n_cls] = obj_feats[N, C] * proto[n_cls, C]^T     (matching_baseline_utils.py:896)
//
// D[M, N] (fp32) = A[M, K'] * B[N, K']^T with bf16 operands, K-major, staged by TMA into 128B-swizzled shared
// memory and multiplied by tcgen05.mma (cta_group::1, UMMA 128 x BN x 16) into a TMEM accumulator.
//
// fp32 accuracy on bf16 tensor cores: each fp32 operand x is split into hi = bf16(x), lo = bf16(x - hi) and the
// three significant partial products are laid side by side along K,
//     A' = [A_hi | A_hi | A_lo],  B' = [B_hi | B_lo | B_hi]   =>   A'B'^T = A_hi B_hi + A_hi B_lo + A_lo B_hi,
// so one ordinary bf16 GEMM with K' = 3*Kp yields ~2^-17 relative error (the dropped lo*lo term), far inside
// the 1e-3 parity bound and small enough not to disturb score rankings.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one elected lane),
// warps 2..5 = epilogue (TMEM -> registers -> global), one TMEM lane quarter each.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace nttt {

constexpr int kBM = 128;      // UMMA_M
constexpr int kBK = 64;       // bf16 elements per k-block = 128 bytes = one swizzle atom row
constexpr int kUmmaK = 16;    // bf16
constexpr int kGemmThreads = 192;

// ---------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a lost arrive traps (CUDA error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// K-major, 128-byte swizzle: atoms of 8 rows x 128 B, SBO = 1024 B between 8-row groups, LBO unused
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);        // start address, bits [0,14)
  d |= (uint64_t)0 << 16;                             // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                   // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                             // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                             // layout type: SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=bn
__host__ __device__ constexpr uint32_t umma_idesc(int bn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
      "%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// epilogue warps 2..5: TMEM lane quarter q = warp % 4 -> registers -> global
template <int BN>
__device__ __forceinline__ void gemm_epilogue(uint32_t tmem_acc, uint64_t* acc_ready, int q, int lane, int m0, int n0,
                                              float* __restrict__ D, int ldd, int M, int N) {
  mbar_wait(acc_ready, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int row = m0 + q * 32 + lane;
#pragma unroll
  for (int cb = 0; cb < BN; cb += 32) {
    uint32_t r[32];
    tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + cb, r);
    if (row < M) {
      float* dst = D + (size_t)row * ldd + n0 + cb;
      if (n0 + cb + 32 <= N && (ldd & 3) == 0) {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                             __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (n0 + cb + j < N) dst[j] = __uint_as_float(r[j]);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// the kernel: one CTA per 128 x BN output tile
// ---------------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct GemmSmem {
  alignas(1024) __nv_bfloat16 a[STAGES][kBM * kBK];
  alignas(1024) __nv_bfloat16 b[STAGES][BN * kBK];
  alignas(8) uint64_t full[STAGES];
  alignas(8) uint64_t empty[STAGES];
  alignas(8) uint64_t acc_ready;
  uint32_t tmem_base;
  uint32_t act;  // k-blocks of one operand segment that this tile has to multiply (skipping mode)
};

// kBank (nttt_match_image_banked, similarity launches): N is the bank's capacity; the live column count is read from
// *bank (bank_rows), and tiles that lie wholly at or past it exit before they allocate TMEM or issue a TMA or an MMA.
// kCounted (nttt_match_image_counted): M is the candidate capacity; the live row count is read from *live.n, row tiles
// wholly at or past it exit the same way, and the epilogue (and the k-block skip mask) stop at it.  With live.split_sm
// the split-K is the one the low-latency mode picks at the live count: the grid holds the largest split (one row tile),
// the k-blocks per split follow the live count, the z-slices past its partials exit, and the partials are k * ldd
// floats apart, so that top1_kernel<.., true> adds exactly the partials nttt_match_image adds at that count.
template <int BN, int STAGES, bool kBank, bool kCounted>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               float* __restrict__ D, int ldd, int M, int N, int total_k_blocks, int kb_per_split,
               size_t split_stride, const uint32_t* __restrict__ a_active, const uint8_t* __restrict__ b_nonfinite,
               int nkb_seg, const nttt_match_bank* __restrict__ bank, int bank_neg, LiveCount live) {
  // Skipping mode (a_active != nullptr; no split-K): K' is nseg = total_k_blocks / nkb_seg segments of nkb_seg k-blocks
  // (the split-bf16 layout: 3), a_active[row] has bit kb set if row `row` of A holds anything but zeros in k-block kb of a
  // segment, b_nonfinite[r-tile * nkb_seg + kb] is 1 if rows 32 r-tile .. +31 of B hold an inf / NaN there.  A k-block in
  // which all 128 rows of the A tile are zero and the B tile is finite adds exact zeros: it is neither loaded nor
  // multiplied.  (The pooling operand is a mask's projection onto the encoder grid: a quarter of the k-blocks per mask.)
  extern __shared__ uint8_t smem_raw[];
  auto& sm = *reinterpret_cast<GemmSmem<BN, STAGES>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * BN;
  if constexpr (kBank) {
    // (the struct is read once the predecessor has completed: this instance does not overlap its set-up with the drain)
    chain_wait();
    if (n0 >= bank_rows(bank, bank_neg)) return;
  }
  if constexpr (kCounted) {
    // (read without waiting for the predecessor: the count is written before the stage's first kernel, an ordinary
    // launch, so this instance still sets up its barriers and TMEM while the producer of the operands drains.  A CTA
    // that exits still waits first: chain_wait is on every path, so the kernels after this one stay ordered behind all
    // earlier ones.)
    M = live_count(live);
    bool idle = m0 >= M;
    if (!idle && live.split_sm > 0) {
      kb_per_split = split_kb_per(live.split_k, sim_split_want(M, N, live.split_k, live.split_sm));
      idle = (int)blockIdx.z * kb_per_split >= total_k_blocks;
      split_stride = (size_t)M * ldd;
    }
    if (idle) {
      chain_wait();
      return;
    }
  }
  // split-K: blockIdx.z owns k-blocks [kb0, kb0 + num_k_blocks) and writes its partial tile to D + z*split_stride
  const int kb0 = blockIdx.z * kb_per_split;
  const int num_k_blocks = min(kb_per_split, total_k_blocks - kb0);
  D += (size_t)blockIdx.z * split_stride;
  constexpr uint32_t kStageBytes = (kBM + BN) * kBK * sizeof(__nv_bfloat16);
  constexpr uint32_t kTmemCols = BN < 32 ? 32 : BN;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
    for (int s = 0; s < STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
    mbar_init(&sm.acc_ready, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)),
                 "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_acc = sm.tmem_base;
  chain_wait();  // (barriers, TMEM and tensor-map prefetch are set up while the producer of the operands drains)

  const bool skipping = a_active != nullptr && nkb_seg > 0 && nkb_seg <= 32 && gridDim.z == 1;
  uint32_t act = 0;
  if (skipping) {
    if (threadIdx.x == 0) sm.act = 0u;
    __syncthreads();
    uint32_t m = 0;
    for (int r = threadIdx.x; r < kBM && m0 + r < M; r += kGemmThreads) m |= a_active[m0 + r];
    if (b_nonfinite) {
      const int rt0 = n0 >> 5, rt1 = min((n0 + BN + 31) >> 5, (N + 31) >> 5);
      for (int i = threadIdx.x; i < (rt1 - rt0) * nkb_seg; i += kGemmThreads) {
        const int rt = rt0 + i / nkb_seg, kb = i - (i / nkb_seg) * nkb_seg;
        if (b_nonfinite[rt * nkb_seg + kb]) m |= 1u << kb;
      }
    }
    m = __reduce_or_sync(0xffffffffu, m);
    if (lane == 0 && m) atomicOr(&sm.act, m);
    __syncthreads();
    act = sm.act & (nkb_seg >= 32 ? 0xffffffffu : ((1u << nkb_seg) - 1u));
    if (act == 0u) act = 1u;  // (an all-zero tile still has to write its zeros)
  }
  const int per_seg = skipping ? __popc(act) : 0;
  const int n_exec = skipping ? per_seg * (total_k_blocks / nkb_seg) : num_k_blocks;
  // global k-block index of the it-th executed one
  auto kb_index = [&](int it) -> int {
    if (!skipping) return kb0 + it;
    const int seg = it / per_seg;
    return seg * nkb_seg + (int)__fns(act, 0, it - seg * per_seg + 1);
  };

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < n_exec; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        const int col = kb_index(kb) * kBK;
        mbar_wait(&sm.empty[s], ph ^ 1);
        mbar_expect_tx(&sm.full[s], kStageBytes);
        tma_load_2d(sm.a[s], &map_a, &sm.full[s], col, m0);
        tma_load_2d(sm.b[s], &map_b, &sm.full[s], col, n0);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(BN);
      for (int kb = 0; kb < n_exec; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(&sm.full[s], ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_addr = smem_u32(sm.a[s]), b_addr = smem_u32(sm.b[s]);
#pragma unroll
        for (int k = 0; k < kBK / kUmmaK; ++k) {
          const uint64_t ad = umma_smem_desc(a_addr + k * kUmmaK * 2);
          const uint64_t bd = umma_smem_desc(b_addr + k * kUmmaK * 2);
          umma_f16(tmem_acc, ad, bd, idesc, (kb | k) != 0);
        }
        umma_commit(&sm.empty[s]);  // frees the smem slot once these MMAs have read it
      }
      umma_commit(&sm.acc_ready);   // accumulator complete
    }
  } else {
    gemm_epilogue<BN>(tmem_acc, &sm.acc_ready, warp & 3, lane, m0, n0, D, ldd, M, N);
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(kTmemCols));
  }
}

// ---------------------------------------------------------------------------------------------------
// host: tensor maps + launch
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// row-major bf16 [rows, k] with k contiguous; box = [box_rows, 64]
static int make_map(CUtensorMap* map, const void* base, int rows, int k, int ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return NTTT_ECUDA;
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(__nv_bfloat16)};
  cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    cuda_fail(cudaErrorInvalidValue, "cuTensorMapEncodeTiled");
    return NTTT_ECUDA;
  }
  return NTTT_OK;
}

template <int BN, int STAGES>
static int launch_tc(const __nv_bfloat16* A, int lda, const __nv_bfloat16* B, int ldb, float* D, int ldd, int M, int N,
                     int K, int splits, size_t split_stride, cudaStream_t s, const uint32_t* a_active,
                     const uint8_t* b_nonfinite, const nttt_match_bank* bank, int bank_neg, const LiveCount* live) {
  CUtensorMap ma, mb;
  int err = make_map(&ma, A, M, K, lda, kBM);
  if (err) return err;
  err = make_map(&mb, B, N, K, ldb, BN);
  if (err) return err;
  const size_t smem = sizeof(GemmSmem<BN, STAGES>) + 1024;
  auto kern = live ? (bank ? gemm_tc_kernel<BN, STAGES, true, true> : gemm_tc_kernel<BN, STAGES, false, true>)
                   : (bank ? gemm_tc_kernel<BN, STAGES, true, false> : gemm_tc_kernel<BN, STAGES, false, false>);
  NTTT_CUDA(set_dyn_smem(kern, (int)smem));
  const int total_kb = K / kBK;
  const int kb_per = ceil_div(total_kb, splits);
  dim3 grid(ceil_div(N, BN), ceil_div(M, kBM), ceil_div(total_kb, kb_per));
  const int nkb_seg = (a_active && K % (3 * kBK) == 0) ? K / 3 / kBK : 0;
  launch_chain(kern, grid, kGemmThreads, smem, s, ma, mb, D, ldd, M, N, total_kb, kb_per, split_stride, a_active, b_nonfinite,
               nkb_seg, bank, bank_neg, live ? *live : LiveCount{});
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// A [M, K] and B [N, K] bf16, K a multiple of 64, rows 16-byte aligned (lda, ldb multiples of 8)
// splits > 1: split-K, partial tile z is written to D + z*split_stride (the caller sums the partials in a fixed
// order); *splits_out receives the number of partials actually produced.
// bank (nullable): B is a bound bank's split prototype table of N (the capacity) rows, of which bank_rows(bank, bank_neg)
// are live; the tiles past them are not computed (gemm_tc_kernel<.., true, ..>).
// live (nullable): M is the capacity of a counted call, the live row count is read on the device (gemm_tc_kernel<.., true>);
// with live->split_sm, `splits` is the largest split the live count can take and *splits_out is not meaningful.
int launch_gemm_tc(const void* A, int lda, const void* B, int ldb, float* D, int ldd, int M, int N, int K, int splits,
                   size_t split_stride, int* splits_out, cudaStream_t s, bool low_latency, const uint32_t* a_active,
                   const uint8_t* b_nonfinite, const nttt_match_bank* bank, int bank_neg, const LiveCount* live) {
  if (splits_out) *splits_out = 1;
  if (M <= 0 || N <= 0) return NTTT_OK;
  if (K <= 0 || K % kBK != 0 || lda % 8 != 0 || ldb % 8 != 0 || splits < 1) return NTTT_EINVAL;
  const int total_kb = K / kBK;
  const int kb_per = ceil_div(total_kb, splits);
  if (splits_out) *splits_out = ceil_div(total_kb, kb_per);
  const __nv_bfloat16* a = static_cast<const __nv_bfloat16*>(A);
  const __nv_bfloat16* b = static_cast<const __nv_bfloat16*>(B);
  // wide outputs (the pooling GEMM, N = C) use 128 x 128 tiles: the kernel is bound by L2 -> shared-memory operand
  // traffic, which scales with 1/BM + 1/BN; narrow outputs (similarity, N = n_cls) keep 128 x 64 for more CTAs
  // 128 x 256 tiles halve the CTA count and raise the flops per operand byte by a third.  With many images in flight
  // the stage's throughput follows the SM-time a kernel consumes, not its latency: 32 CTAs x 38 us beat 64 CTAs x 25 us
  // at 1024 rows (97.9 vs 100.3 us/image), and at 4096 rows one wave of 128 CTAs beats 1.7 waves of 256 (281 vs 292).
  // (N need not be a multiple of 256: TMA zero-fills the rows past N and the epilogue bounds its stores)
  // The 128 x 256 kernel is tensor-pipe bound, so three 48 KB stages feed it as well as four and leave 83 KB of the SM's
  // shared memory to CTAs of the other kernels of the images in flight (measured 91.8 vs 92.3 us/image; two stages: 92.0).
  const bool bn256 = !low_latency && N >= 512 && M >= 512;
  const bool bn128 = N >= 512 || (N > 64 && N <= 128);  // 65..128 columns: ONE 128-wide tile reads the A operand once instead of twice
  if (bn256)
    return launch_tc<256, 3>(a, lda, b, ldb, D, ldd, M, N, K, splits, split_stride, s, a_active, b_nonfinite, bank, bank_neg,
                                  live);
  if (bn128)
    return launch_tc<128, 5>(a, lda, b, ldb, D, ldd, M, N, K, splits, split_stride, s, a_active, b_nonfinite, bank, bank_neg,
                                  live);
  return launch_tc<64, 6>(a, lda, b, ldb, D, ldd, M, N, K, splits, split_stride, s, a_active, b_nonfinite, bank, bank_neg,
                                  live);
}

// ---------------------------------------------------------------------------------------------------
// operand preparation: fp32 -> split bf16, three K-segments of width kp (zero padded)
//   mode 0 (A operand): [hi | hi | lo]      mode 1 (B operand): [hi | lo | hi]
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// kBank (nttt_match_image_banked): X is the bound bank's prototype table (bank->proto, or bank->proto_neg when bank_neg)
// and `rows` its capacity; rows from the live count (bank_rows) up to the capacity are written as zeros, so that no GEMM
// tile reads the rows of a bank bound before
template <bool kBank>
__global__ void __launch_bounds__(256)
split_rows_kernel(const float* __restrict__ X, int ld, int rows, int k, int kp, int mode,
                  __nv_bfloat16* __restrict__ out, const nttt_match_bank* __restrict__ bank, int bank_neg) {
  const int r = blockIdx.y;
  bool live = true;
  if constexpr (kBank) {
    X = bank_neg ? bank->proto_neg : bank->proto;
    live = r < bank_rows(bank, bank_neg);
  }
  const float* src = X + (size_t)r * ld;
  __nv_bfloat16* dst = out + (size_t)r * 3 * kp;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kp; i += gridDim.x * blockDim.x) {
    __nv_bfloat16 hi = __float2bfloat16_rn(0.0f), lo = hi;
    if (i < k && live) split_bf16(src[i], hi, lo);
    dst[i] = hi;
    dst[kp + i] = mode == 0 ? hi : lo;
    dst[2 * kp + i] = mode == 0 ? lo : hi;
  }
}

// X [k, rows] (row-major, ld) -> out [rows, 3*kp]: transpose + split (for feat [E, C] -> [C, 3*Ep]).
// 64 (k) x 32 (rows) tiles: 128-byte coalesced reads along `rows`, and every thread writes two consecutive k as one
// bf16x2, so a warp stores 128 contiguous bytes per segment (kp is a multiple of 64).
// (A function of its own: written inside the kernel, these statements compile to different SASS; this is the one
// measured.)
__device__ __forceinline__ void split_transpose_body(const float* __restrict__ X, int ld, int rows, int k, int kp, int mode,
                                                     __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ nonfinite) {
  // nonfinite (nullable) [kp / 64, ceil(rows / 32)]: 1 where the tile holds an inf or a NaN — a GEMM that skips k-blocks
  // whose OTHER operand is all zeros must not skip those (0 * inf = NaN in the reference's dense product)
  __shared__ float tile[64][33];
  const int tiles_k = kp / 64, tiles_r = (rows + 31) / 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int tile_id = blockIdx.x; tile_id < tiles_k * tiles_r; tile_id += gridDim.x) {  // (a few tiles per CTA)
    const int k0 = (tile_id % tiles_k) * 64, r0 = (tile_id / tiles_k) * 32;
    if (tile_id != (int)blockIdx.x) __syncthreads();  // the previous tile has been written out
    int bad = 0;
#pragma unroll
    for (int j = ty; j < 64; j += 8) {
      const int kk = k0 + j, rr = r0 + tx;
      const float v = (kk < k && rr < rows) ? X[(size_t)kk * ld + rr] : 0.0f;
      bad |= (__float_as_uint(v) & 0x7f800000u) == 0x7f800000u;
      tile[j][tx] = v;
    }
    bad = __syncthreads_or(bad);
    if (nonfinite && threadIdx.x == 0) nonfinite[tile_id] = (uint8_t)(bad != 0);  // tile_id = r-tile * tiles_k + k-tile
    const int kk = k0 + 2 * tx;
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
      const int rr = r0 + j;
      if (rr < rows && kk + 1 < kp) {
        __nv_bfloat16 h0, l0, h1, l1;
        split_bf16(tile[2 * tx][j], h0, l0);
        split_bf16(tile[2 * tx + 1][j], h1, l1);
        const __nv_bfloat162 hi = __halves2bfloat162(h0, h1), lo = __halves2bfloat162(l0, l1);
        __nv_bfloat16* dst = out + (size_t)rr * 3 * kp + kk;
        *reinterpret_cast<__nv_bfloat162*>(dst) = hi;
        *reinterpret_cast<__nv_bfloat162*>(dst + kp) = mode == 0 ? hi : lo;
        *reinterpret_cast<__nv_bfloat162*>(dst + 2 * kp) = mode == 0 ? lo : hi;
      }
    }
  }
}

// kBound (nttt_match_image_bound): X's address is read from *x_at (nttt_match_inputs.tar_feat) instead
template <bool kBound>
__global__ void __launch_bounds__(256)
split_transpose_kernel(const float* __restrict__ X, int ld, int rows, int k, int kp, int mode,
                       __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ nonfinite,
                       const float* const* __restrict__ x_at) {
  split_transpose_body(kBound ? *x_at : X, ld, rows, k, kp, mode, out, nonfinite);
}

// bank (nullable): split the bound bank's table (X is then ignored; rows = the capacity)
int launch_split_rows(const float* X, int ld, int rows, int k, int kp, int mode, void* out, cudaStream_t s,
                      const nttt_match_bank* bank, int bank_neg) {
  if (rows <= 0) return NTTT_OK;
  dim3 grid(ceil_div(kp, 256), rows);
  (bank ? split_rows_kernel<true> : split_rows_kernel<false>)<<<grid, 256, 0, s>>>(
      X, ld, rows, k, kp, mode, static_cast<__nv_bfloat16*>(out), bank, bank_neg);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

// x_at (nullable): read X's address from device memory when the kernel runs (X is then ignored)
int launch_split_transpose(const float* X, int ld, int rows, int k, int kp, int mode, void* out, cudaStream_t s,
                           uint8_t* nonfinite, const float* const* x_at) {
  if (rows <= 0) return NTTT_OK;
  if (kp % 64 != 0) return NTTT_EINVAL;  // (callers pad K to 64: the GEMM's K block)
  const int tiles = (kp / 64) * ceil_div(rows, 32);
  const int grid = t_low_latency ? tiles : min(tiles, 148);
  (x_at ? split_transpose_kernel<true> : split_transpose_kernel<false>)<<<grid, 256, 0, s>>>(
      X, ld, rows, k, kp, mode, static_cast<__nv_bfloat16*>(out), nonfinite, x_at);
  NTTT_LAUNCH_CHECK();
  return NTTT_OK;
}

}  // namespace nttt
