// Shared device/host helpers for libnttt_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/nttt_b200.h"

namespace nttt {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// launch-site error capture: records the CUDA error text for nttt_last_cuda_error()
int cuda_fail(cudaError_t e, const char* what);
#define NTTT_CUDA(expr)                                        \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) return ::nttt::cuda_fail(_e, #expr); \
  } while (0)
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (device, kernel, size reached): the call costs several
// microseconds of host time, which a caller that launches one image at a time pays on every kernel
cudaError_t set_dyn_smem_impl(const void* fn, int bytes);
template <typename F>
inline cudaError_t set_dyn_smem(F* fn, int bytes) { return set_dyn_smem_impl(reinterpret_cast<const void*>(fn), bytes); }
// every kernel launch of the library passes through here; the counter backs nttt_launch_count()
// Set by nttt_match_image for the duration of the call (launchers run on the calling thread): kernels take the launch
// shape with the shortest duration of ONE image instead of the thin persistent shape that costs the least when many
// images are in flight (nttt_match_args.low_latency).  Results do not depend on it.
extern thread_local bool t_low_latency;
// set after a cross-stream event wait: the next chain launch is an ordinary one (its predecessor in the stream is the
// wait, not a kernel that triggers), then the flag clears itself
extern thread_local bool t_chain_break;
extern std::atomic<unsigned long long> g_launches;  // (host threads of different contexts may launch concurrently)
#define NTTT_LAUNCH_CHECK()          \
  do {                               \
    ++::nttt::g_launches;            \
    NTTT_CUDA(cudaGetLastError());   \
  } while (0)

// Launch of a kernel on the main chain of nttt_match_image.  In low-latency mode (one image at a time) the launch carries
// the programmatic-stream-serialization attribute: the kernel may be scheduled while its predecessor's last CTAs are
// still running, and its `chain_wait()` — the first statement of every chain kernel — holds it until the predecessor
// has completed and its writes are visible.  What overlaps is the launch latency and the CTA ramp-up, 2-3 us per kernel
// boundary of an 18-kernel chain.  Without the attribute (many images in flight: other streams fill the gaps anyway)
// chain_wait() returns immediately.
template <typename... KArgs, typename... Args>
inline void launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (t_low_latency && !t_chain_break) ? 1 : 0;
  t_chain_break = false;
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // (the error is picked up by NTTT_LAUNCH_CHECK)
}
#ifdef __CUDACC__
// first statement of every chain kernel, in every CTA and on every path: wait for the predecessor grid (and, through it,
// for every earlier one), then let the successor be scheduled once all CTAs of this grid have got here
__device__ __forceinline__ void chain_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
#endif

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(kFull, v, o));
  return v;
}

// Bitonic sort of 1024 64-bit keys held one per thread (blockDim.x == 1024), ascending: thread i returns the
// i-th smallest key.  Exchanges at distance < 32 are warp shuffles; only the 15 stages at distance >= 32 go
// through shared memory (s_x: 1024 keys).  Keys must be distinct (callers put the index in the low bits).
__device__ __forceinline__ unsigned long long block_bitonic_sort_1024(unsigned long long key,
                                                                      unsigned long long* s_x) {
  const int i = threadIdx.x;
  for (int k = 2; k <= 1024; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      unsigned long long other;
      if (j >= 32) {
        s_x[i] = key;
        __syncthreads();
        other = s_x[i ^ j];
        __syncthreads();
      } else {
        other = __shfl_xor_sync(kFull, key, j);
      }
      const bool take_min = ((i & j) == 0) == ((i & k) == 0);
      key = (take_min == (other < key)) ? other : key;
    }
  }
  return key;
}

// streaming 128-bit load that does not pollute L1 (data is touched once)
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// ---------------------------------------------------------------------------------------------------
// Antialias (Pillow-style) bilinear weight tables for one axis, shared by the full-res resize kernel
// and the mask projection.  Built on the device with the exact fp32 recipe of aten's
// _upsample_bilinear2d_aa (see DESIGN.md §resize).
// ---------------------------------------------------------------------------------------------------
struct AxisTable {
  int in_size = 0, out_size = 0, taps = 0;
  void* slab = nullptr;      // the one device allocation every array below points into
  int32_t* xmin = nullptr;   // [out]
  int32_t* xsize = nullptr;  // [out]
  float* w = nullptr;        // [out, taps]
  // transposed (scatter) view: for input coordinate e, the contiguous output range whose span holds e
  int32_t* t_lo = nullptr;   // [in]
  int32_t* t_len = nullptr;  // [in]
  float* t_w = nullptr;      // [in, kMaxScatter]
  float* t_cum = nullptr;    // [in, kMaxScatter + 1] running sums of t_w (t_cum[e][0] = 0)
  // output coordinates grouped into runs (<= kGrpMax long) that share the same input span (xmin, xsize):
  // rows of one group read the same input rows, so the horizontal pass and the footprint test are shared
  int32_t* grp_of = nullptr;     // [out]  group index of each output coordinate
  int32_t* grp_start = nullptr;  // [out + 1] first coordinate of each group, grp_start[n_groups] = out
  // two-tap records of the resize fast path, built only when every span has xsize <= 2 (up-scaling, except the sizes
  // where fp32 rounding widens a span to three samples, see aa_spans_within_two; tests/test_resize_two_tap.py): per
  // output coordinate the span {xmin | xsize << 16} and the weights {w0, w1} (w1 = 0 when xsize = 1), padded with
  // all-zero records (xsize = 0) up to a multiple of 32 coordinates
  uint32_t* pk_span = nullptr;   // [align32(out)] or nullptr
  float2* pk_w = nullptr;        // [align32(out)] or nullptr
};
constexpr int kGrpMax = 4;
constexpr int kMaxScatter = 24;

int aa_max_taps(int in_size, int out_size);

// base pointers of the decoder's per-batch output tensors, passed to multimask_select_kernel BY VALUE (stream-ordered,
// graph-capturable, no staging copy)
constexpr int kMaxChunks = 64;
static_assert(kMaxChunks == NTTT_MAX_CHUNKS, "the bound inputs hold as many chunks as the by-value table");
struct ChunkTable {
  const float* base[kMaxChunks];
};

// internal launchers (defined in the .cu files, called by api.cu)
int build_axis_table(AxisTable& t, int in_size, int out_size, cudaStream_t s);
void free_axis_table(AxisTable& t);

// ---------------------------------------------------------------------------------------------------
// Sized entry (nttt_match_image_sized): the output size is read from device memory when the kernels run, within a range
// [min, capacity] fixed when the call is enqueued.  The resize tables of every size of the range come from an ATLAS,
// built once per (low-res size, range) and owned by the context: one slab holding, per axis and output size, the
// AxisTable arrays the resize reads (no scatter view), and a device index of SizedAxis records.
// ---------------------------------------------------------------------------------------------------
struct SizedAxis {  // one output size of one axis
  const int32_t* xmin; const int32_t* xsize; const float* w;
  const int32_t* t_lo; const int32_t* t_len; const int32_t* grp_of; const int32_t* grp_start;
  const uint32_t* pk_span; const float2* pk_w;  // nullptr: the size takes the general resize path on this axis
  int taps;
  int budget;  // this axis's factor of the two-tap resize's logit tile budget (up2_tile_factor)
};
// by-value kernel argument that every kernel depending on the output size takes after its static parameters: read only
// by the kernel's kSized = true instance (the static instance is passed an empty one)
struct SizedDims {
  const int32_t* hw;      // [2] (h, w), device
  const SizedAxis* ay;    // [cap_h - min_h + 1] output heights
  const SizedAxis* ax;    // [cap_w - min_w + 1] output widths
  int32_t* counts;        // nttt_match_args.counts: [1] emptied and [3] (status) written by the resize
  int min_h, min_w, cap_h, cap_w;
};
struct SizedAtlas {
  int lr_h = 0, lr_w = 0, min_h = 0, min_w = 0, cap_h = 0, cap_w = 0;
  char* slab = nullptr;
  size_t bytes = 0;
  double build_ms = 0.0;  // host time of the build, behind its one stream synchronisation
  SizedAxis* ay = nullptr;  // device index (inside the slab)
  SizedAxis* ax = nullptr;
  bool any_two_tap = false;  // some size of the range takes the two-tap resize on both axes
  bool any_general = false;  // some size takes the general resize
  long max_budget = 0;       // the largest tile budget over the range (sizes the two-tap resize's shared memory)
};
int build_sized_atlas(SizedAtlas& a, cudaStream_t s);  // a: sizes set; fills the rest (one synchronisation)
long up2_tile_factor(int in_size, int out_size, bool rows);

#ifdef __CUDACC__
// (h, w) of this call; a size outside the range reads as the capacity and returns false
__device__ __forceinline__ bool sized_hw(const SizedDims& d, int& h, int& w) {
  h = d.hw[0];
  w = d.hw[1];
  if (h >= d.min_h && h <= d.cap_h && w >= d.min_w && w <= d.cap_w) return true;
  h = d.cap_h;
  w = d.cap_w;
  return false;
}
#endif

}  // namespace nttt

struct nttt_ctx {
  int device = 0;
  int sm_count = 0;
  // cache of antialias tables keyed by (in,out); least-recently-used entry of an EARLIER call is evicted.  An image
  // takes two tables keyed by its height and its width (COCO / LVIS: a few hundred distinct values each), so the cache
  // holds 1024 of them (~100 KB each); evicted tables are only RETIRED — kernels of earlier calls on other streams may
  // still read them — and the retired ones are freed in batches behind one device synchronisation.
  static constexpr int kMaxTables = 1024;
  static constexpr int kMaxRetired = 64;
  nttt::AxisTable tables[kMaxTables];
  unsigned long long last_use[kMaxTables] = {};
  nttt::AxisTable retired[kMaxRetired];
  int n_retired = 0;
  int max_tables = kMaxTables;  // nttt_ctx_tune(NTTT_TUNE_AXIS_CACHE_ENTRIES): smaller caches for tests
  unsigned long long epoch = 0;  // bumped once per API call that takes tables
  int n_tables = 0;
  // shared-memory budget of upsample_pack's logit tile, in floats (nttt_ctx_tune; 0 = read taps from global memory)
  int upsample_stage_floats = 36 * 1024 / 4;
  // nttt_ctx_tune(NTTT_TUNE_POOL_ORDER): 0 runs the pooling GEMM of nttt_match_image on unordered rows (the path of
  // the low-latency mode and of n <= 128), so that tests can compare it with the ordered one
  bool pool_order = true;
  int32_t* scratch = nullptr;  // per-mask statistics scratch of the stand-alone resize entry
  size_t scratch_cap = 0;  // bytes
  // optional per-stage CUDA-event profile of nttt_match_image (off by default)
  static constexpr int kMaxStages = 16;
  bool profile = false;
  int stop_after = 0;  // debugging/profiling: stop nttt_match_image after this many stages (0 = run all)
  cudaEvent_t ev[kMaxStages + 1] = {};
  int n_ev = 0;
  // side stream of the low-latency mode (created on first use; the context is not thread-safe, see the header)
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool side_ready() {
    if (side) return true;
    if (cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking) != cudaSuccess) { side = nullptr; return false; }
    if (cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) != cudaSuccess) {
      cudaStreamDestroy(side);
      side = nullptr;
      return false;
    }
    return true;
  }
  // returns the table BY VALUE (device pointers stay valid until evicted by a later call)
  int axis(int in_size, int out_size, cudaStream_t s, nttt::AxisTable* out);
  // atlases of the sized entry, one per (low-res size, range); kept until the context is destroyed (graphs captured
  // with one keep reading it)
  static constexpr int kMaxAtlases = 16;
  nttt::SizedAtlas atlases[kMaxAtlases];
  int n_atlases = 0;
  int sized_atlas(int lr_h, int lr_w, int min_h, int min_w, int cap_h, int cap_w, cudaStream_t s,
                  const nttt::SizedAtlas** out);
};
