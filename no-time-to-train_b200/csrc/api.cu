// C-ABI of libnttt_b200.so (see include/nttt_b200.h).  Host-side only: argument checks, workspace carving,
// kernel launches.  No allocation per call, no device synchronisation (except one-time table builds).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace nttt {

// launchers implemented in the kernel translation units
int launch_lowres_pack(const float*, int, int, int, float, float, uint32_t*, int32_t*, int32_t*, int32_t*, int32_t*,
                       const float*, float, const float* const*, cudaStream_t, float* stab_score = nullptr);
int launch_multimask_select(const float*, int, int, int, const ChunkTable&, int, size_t, const float**, float*,
                            cudaStream_t, const float* const* ious_at = nullptr, const float* const* bases = nullptr);
int launch_plane_resolve(const nttt_match_inputs*, int, size_t, const float**, float*, cudaStream_t);
int launch_match_bind(const nttt_match_inputs&, nttt_match_inputs*, cudaStream_t);
int launch_project_masks(const AxisTable&, const AxisTable&, const uint32_t*, const int32_t*, int, int, int, int, int,
                         void*, int, bool, cudaStream_t, const int32_t* perm = nullptr, uint32_t* active = nullptr);
int launch_pool_order(const int32_t*, int, int, int32_t*, cudaStream_t);
int launch_normalize_split(const float*, int, const int32_t*, int, int, int, float*, void*, bool, cudaStream_t,
                           const int32_t* perm = nullptr);
int launch_gemm_tc(const void*, int, const void*, int, float*, int, int, int, int, int, size_t, int*, cudaStream_t,
                   bool low_latency = false, const uint32_t* a_active = nullptr, const uint8_t* b_nonfinite = nullptr);
int gemm_tc_pick_splits(int, int, int, int);
int launch_split_rows(const float*, int, int, int, int, int, void*, cudaStream_t);
int launch_split_transpose(const float*, int, int, int, int, int, void*, cudaStream_t, uint8_t* nonfinite = nullptr,
                           const float* const* x_at = nullptr);
int launch_normalize_rows(const float*, int, const int32_t*, int, int, float*, bool, cudaStream_t);
int launch_proto_prepare(const float*, int, int, int, float*, cudaStream_t);
int launch_top1(const float*, int, size_t, float*, int, int, int, float*, int32_t*, cudaStream_t);
int launch_neg_top1(const float*, int, size_t, const float*, int, size_t, int, int, int, float, float*, float*, int32_t*,
                    cudaStream_t);
size_t nms_workspace_bytes(int n);
int launch_box_nms(const int32_t*, const float*, const int32_t*, const float*, int, float, int, int32_t*, int32_t*,
                   int32_t*, int32_t*, void*, size_t, float, int, cudaStream_t);
int launch_upsample_pack(const AxisTable&, const AxisTable&, const float*, const uint32_t*, const int32_t*,
                         const int32_t*, int, int, const int32_t*, const int32_t*, int, int, int, uint32_t*, int32_t*,
                         int32_t*, int32_t*, int32_t*, const float* const*, cudaStream_t, int, int, uint32_t* bits_t = nullptr,
                         bool* wrote_t = nullptr, bool low_latency = false, int32_t* zero2 = nullptr,
                         const SizedDims* sized = nullptr, const SizedAtlas* atlas = nullptr);
int32_t* ios_pair_counters(void* ws, int max_sel);
size_t upsample_scratch_bytes(int max_sel, int oh, int ow);
int launch_unpack_sparse(const uint32_t*, const int32_t*, const int32_t*, const int32_t*, int, int, int, uint8_t*,
                         int32_t*, cudaStream_t, bool tr = false, const SizedDims* sized = nullptr);
int launch_unpack(const uint32_t*, const int32_t*, const int32_t*, const int32_t*, int, int, int, uint8_t*,
                  cudaStream_t, bool tr = false, const SizedDims* sized = nullptr);
size_t ios_workspace_bytes(int max_sel);
int launch_mask_ios(const uint32_t*, const int32_t*, const int32_t*, const int32_t*, const int32_t*, const int32_t*,
                    int, int, int, const int32_t*, const float*, int, float*, int32_t*, void*, bool, cudaStream_t,
                    const uint32_t* bits_t = nullptr, bool counters_zeroed = false, const SizedDims* sized = nullptr);
int launch_decay_rank(const float*, const int32_t*, const float*, const int32_t*, const int32_t*, int, int,
                      const int32_t*, const int32_t*, int64_t*, float*, int64_t*, int32_t*, int32_t*, int32_t*, float*,
                      cudaStream_t);
int launch_rle_encode(const uint32_t*, const int32_t*, const int32_t*, const int32_t*, int, int, int, int, int, uint32_t*,
                      int32_t*, uint8_t*, int32_t*, cudaStream_t, bool tr = false, const SizedDims* sized = nullptr);
int launch_rle_compact(const uint8_t*, const int32_t*, int, int, uint8_t*, long long, cudaStream_t);
int launch_fill_pool(const float*, const float*, int, int, int, int, int, int, float*, float*, float*, int, cudaStream_t);
int launch_fill_scatter(const float*, const float*, const float*, const int32_t*, int, int, int, float*, float*, float*,
                        cudaStream_t);
int launch_fill_finalize(const float*, const float*, int, int, int, float*, float*, cudaStream_t);

extern int g_pack_persistent;  // lowres.cu
static thread_local char g_cuda_err[512] = "";
std::atomic<unsigned long long> g_launches{0};
thread_local bool t_low_latency = false;
thread_local bool t_chain_break = false;

cudaError_t set_dyn_smem_impl(const void* fn, int bytes) {
  struct Entry { const void* fn; int dev; int bytes; };
  static std::mutex mu;
  static Entry table[256];
  static int n = 0;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  Entry* hit = nullptr;
  for (int i = 0; i < n; ++i)
    if (table[i].fn == fn && table[i].dev == dev) { hit = &table[i]; break; }
  if (hit && hit->bytes >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  if (hit) hit->bytes = bytes;
  else if (n < 256) table[n++] = Entry{fn, dev, bytes};
  return cudaSuccess;
}

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? NTTT_ENODEVICE : NTTT_ECUDA;
}

// bump allocator over the caller's workspace
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += sizeof(T) * count;
    return p;
  }
};

inline int pad64(int k) { return (k + 63) / 64 * 64; }

// sums[n, c] = proj[n, e] * feat[e, c] on the tensor cores (split-bf16, K' = 3 * pad64(e))
// scratch: a_split [n, 3*ep] bf16, b_split [c, 3*ep] bf16
// (proj == nullptr: a_split already holds the split projection, written by project_masks_kernel<true>)
// The 128 x 128 output tiles of a 1024 x 1024 pooling GEMM occupy 64 of the 148 SMs, each pulling its operands through
// its own L2 port: split K in kPoolSplits so that twice as many SMs share the same traffic.  The partial sums go to
// sums[z] (stride n*c floats) and are added in a fixed order by the normalisation kernel that reads them anyway.
constexpr int kPoolSplitsMax = 2;  // workspace is sized for the low-latency mode
constexpr int kPoolSplits = 1;  // measured: 2 halves the latency (25 -> 14 us) but costs throughput (100.7 -> 103.5 us/image with 16 images in flight: more SM-time in total)
// low_latency (nttt_match_args.low_latency): one image at a time with a host synchronisation behind it — what counts
// is the duration of each kernel, so the pooling GEMM spreads over twice the SMs (128 x 128 tiles, split-K 2: 14 us
// instead of 25-38 us).
static int pool_contract(const float* proj, const float* feat, int n, int e, int c, float* sums, void* a_split,
                         void* b_split, int* n_partials, cudaStream_t s, bool low_latency = false, bool b_ready = false,
                         const uint32_t* a_active = nullptr, uint8_t* b_nonfinite = nullptr,
                         const float* const* feat_at = nullptr) {
  // a_active / b_nonfinite (both or neither): the A operand's rows are spatially ordered and carry their non-zero k-block
  // masks; the GEMM skips the k-blocks a tile does not touch (gemm_tc_kernel), unless the features are not finite there
  // feat_at (nullable): the features' address is read from device memory when the kernel runs (bound inputs)
  const int ep = pad64(e);
  int err = proj ? launch_split_rows(proj, e, n, e, ep, 0, a_split, s) : NTTT_OK;
  if (err) return err;
  err = b_ready ? NTTT_OK : launch_split_transpose(feat, c, c, e, ep, 1, b_split, s, a_active ? b_nonfinite : nullptr,
                                                   feat_at);  // (b_ready: done on the side stream)
  if (err) return err;
  return launch_gemm_tc(a_split, 3 * ep, b_split, 3 * ep, sums, c, n, c, 3 * ep, low_latency ? kPoolSplitsMax : kPoolSplits,
                        (size_t)n * c, n_partials, s, low_latency, a_active, a_active ? b_nonfinite : nullptr);
}

// rows of `sums` -> /area -> L2-normalise -> obj_feats (+ split-bf16 copy when the vector path applies).
// Returns through *split_done whether a_split now holds the similarity GEMM's A operand.
// nan_empty: negative-reference scoring divides by the raw area (empty mask -> NaN row, as the reference does)
// n_partials: split-K partial sums of the pooling GEMM, n*c floats apart, added in order
static int normalize_rows(const float* sums, int n_partials, const int32_t* area, int n, int c, float* obj_feats,
                          void* a_split, bool* split_done, bool nan_empty, cudaStream_t s, const int32_t* perm = nullptr) {
  *split_done = a_split &&
                launch_normalize_split(sums, n_partials, area, n, c, pad64(c), obj_feats, a_split, nan_empty, s, perm) == 1;
  if (*split_done) return NTTT_OK;
  if (perm) return NTTT_EINVAL;  // (callers order the rows only when the vector path applies)
  return launch_normalize_rows(sums, n_partials, area, n, c, obj_feats, nan_empty, s);
}

// the scatter tables hold kMaxScatter weights per encoder cell: enough while out/in <= ~11
static bool projection_supported(int in_size, int out_size) {
  return in_size > 0 && 2 * ((out_size + in_size - 1) / in_size) + 2 <= kMaxScatter;
}

// sim[n, n_cls] = obj_feats[n, c] * proto[n_cls, c]^T
// (a_ready: a_split already holds the split obj_feats, written by normalize_split_kernel)
// The similarity GEMM has few output tiles (n_cls is small), so it runs split-K into `partials`
// [splits, n, n_cls]; top1_kernel sums them in a fixed order, writes `sim` (nullable) and the row arg-max.
constexpr int kMaxSimSplits = 8;
// floats needed for the split-K partials of an [n, cols] similarity matrix (sized for a 148-SM part)
static size_t sim_partial_floats(int n, int cols, int c) {
  int sp = gemm_tc_pick_splits(n, cols, 3 * pad64(c), 148);
  if (sp > kMaxSimSplits) sp = kMaxSimSplits;
  return (size_t)sp * n * cols;
}

// proto_neg == nullptr: plain cosine scoring.  Otherwise negative-reference scoring: proto is the normalised
// class-level average, proto_neg [n_cls * l_neg, c] the normalised negative instance averages.
static int sim_top1(const float* obj_feats, const float* proto, const float* proto_neg, int l_neg, float sigma, int n,
                    int c, int n_cls, float* sim, float* partials, float* partials_neg, float* top_score,
                    int32_t* top_label, void* a_split, void* b_split, bool a_ready, int sm_count, cudaStream_t s,
                    void* p_split = nullptr, bool p_ready = false) {
  // p_split (nullable): a buffer of its own for the split prototypes, so that they can be prepared before b_split is free
  // (p_ready: already done, on the side stream of the low-latency mode); without it they go through b_split
  const int cp = pad64(c);
  int err = a_ready ? NTTT_OK : launch_split_rows(obj_feats, c, n, c, cp, 0, a_split, s);
  if (err) return err;
  void* pb = p_split ? p_split : b_split;
  err = p_ready ? NTTT_OK : launch_split_rows(proto, c, n_cls, c, cp, 1, pb, s);
  if (err) return err;
  int want = gemm_tc_pick_splits(n, n_cls, 3 * cp, sm_count < 148 ? sm_count : 148);
  if (want > kMaxSimSplits) want = kMaxSimSplits;
  // with many images in flight the partial tiles of a split-K cost more SM-time (8 x the prologues, epilogues and
  // partial sums) than the one long CTA per tile they shorten: measured 84.0 (no split) / 84.6 (2) / 85.1 (4) / 86.8 (8)
  if (!t_low_latency) want = 1;
  const size_t stride = (size_t)n * n_cls;
  int splits = 1;
  err = launch_gemm_tc(a_split, 3 * cp, pb, 3 * cp, partials, n_cls, n, n_cls, 3 * cp, want, stride, &splits, s);
  if (err) return err;
  if (!proto_neg) return launch_top1(partials, splits, stride, sim, n_cls, n, n_cls, top_score, top_label, s);
  const int cols = n_cls * l_neg;
  err = launch_split_rows(proto_neg, c, cols, c, cp, 1, b_split, s);  // stream-ordered after the GEMM that read b_split
  if (err) return err;
  int want_n = gemm_tc_pick_splits(n, cols, 3 * cp, sm_count < 148 ? sm_count : 148);
  if (want_n > kMaxSimSplits) want_n = kMaxSimSplits;
  if (!t_low_latency) want_n = 1;
  const size_t stride_n = (size_t)n * cols;
  int splits_n = 1;
  err = launch_gemm_tc(a_split, 3 * cp, b_split, 3 * cp, partials_neg, cols, n, cols, 3 * cp, want_n, stride_n, &splits_n,
                       s);
  if (err) return err;
  return launch_neg_top1(partials, splits, stride, partials_neg, splits_n, stride_n, n, n_cls, l_neg, sigma, sim,
                         top_score, top_label, s);
}

}  // namespace nttt

using namespace nttt;

int nttt_ctx::axis(int in_size, int out_size, cudaStream_t s, nttt::AxisTable* out) {
  for (int i = 0; i < n_tables; ++i)
    if (tables[i].in_size == in_size && tables[i].out_size == out_size) {
      last_use[i] = epoch;
      *out = tables[i];
      return NTTT_OK;
    }
  int slot = n_tables;
  if (n_tables >= max_tables) {
    // evict the least recently used table that the current call has not taken.  Kernels of earlier calls (possibly on
    // other streams) may still read it, so it is only retired here; retired tables are freed kMaxRetired at a time
    // behind ONE device synchronisation.
    slot = -1;
    for (int i = 0; i < n_tables; ++i)
      if (last_use[i] < epoch && (slot < 0 || last_use[i] < last_use[slot])) slot = i;
    if (slot < 0) return NTTT_EUNSUPPORTED;
    if (n_retired == kMaxRetired) {
      NTTT_CUDA(cudaDeviceSynchronize());
      for (int i = 0; i < n_retired; ++i) free_axis_table(retired[i]);
      n_retired = 0;
    }
    retired[n_retired++] = tables[slot];
  }
  AxisTable t{};
  int err = build_axis_table(t, in_size, out_size, s);
  if (err != NTTT_OK) { free_axis_table(t); return err; }
  // the tables are read by kernels on any stream afterwards: make them visible once, here
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) { free_axis_table(t); return cuda_fail(e, "axis table build"); }
  tables[slot] = t;
  last_use[slot] = epoch;
  if (slot == n_tables) ++n_tables;
  *out = t;
  return NTTT_OK;
}

int nttt_ctx::sized_atlas(int lr_h, int lr_w, int min_h, int min_w, int cap_h, int cap_w, cudaStream_t s,
                          const nttt::SizedAtlas** out) {
  for (int i = 0; i < n_atlases; ++i) {
    const SizedAtlas& a = atlases[i];
    if (a.lr_h == lr_h && a.lr_w == lr_w && a.min_h == min_h && a.min_w == min_w && a.cap_h == cap_h && a.cap_w == cap_w) {
      *out = &a;
      return NTTT_OK;
    }
  }
  if (n_atlases == kMaxAtlases) return NTTT_EUNSUPPORTED;
  SizedAtlas a;
  a.lr_h = lr_h; a.lr_w = lr_w; a.min_h = min_h; a.min_w = min_w; a.cap_h = cap_h; a.cap_w = cap_w;
  int err = build_sized_atlas(a, s);
  if (err) return err;
  atlases[n_atlases] = a;
  *out = &atlases[n_atlases++];
  return NTTT_OK;
}

extern "C" {

int nttt_version(void) { return NTTT_VERSION; }

int nttt_build_is_ablation(void) {
#ifdef NTTT_ABLATE
  return 1;
#else
  return 0;
#endif
}

size_t nttt_sizeof_match_args(void) { return sizeof(nttt_match_args); }

size_t nttt_sizeof_match_inputs(void) { return sizeof(nttt_match_inputs); }

unsigned long long nttt_launch_count(void) { return g_launches.load(); }

static const char* const kStageNames[] = {"lowres_pack", "project_masks", "pool_gemm", "normalize_rows", "sim_top1",
                                          "box_nms", "upsample_pack", "mask_ios", "decay_rank", "unpack", "rle_encode"};
static constexpr int kNumStages = sizeof(kStageNames) / sizeof(kStageNames[0]);

int nttt_profile_num_stages(void) { return kNumStages; }
const char* nttt_profile_stage_name(int i) { return (i >= 0 && i < kNumStages) ? kStageNames[i] : ""; }

int nttt_ctx_tune(nttt_ctx* ctx, int what, long long value) {
  if (!ctx) return NTTT_EINVAL;
  switch (what) {
    case NTTT_TUNE_AXIS_CACHE_ENTRIES:
      if (value < 8 || value > nttt_ctx::kMaxTables) return NTTT_EINVAL;
      if (value < ctx->n_tables) {  // shrinking below what is held: drop the whole cache (behind a device sync)
        NTTT_CUDA(cudaDeviceSynchronize());
        for (int i = 0; i < ctx->n_tables; ++i) free_axis_table(ctx->tables[i]);
        for (int i = 0; i < ctx->n_retired; ++i) free_axis_table(ctx->retired[i]);
        ctx->n_tables = ctx->n_retired = 0;
      }
      ctx->max_tables = (int)value;
      return NTTT_OK;
    case NTTT_TUNE_LOWRES_PERSISTENT:
      if (value < 0 || value > 1) return NTTT_EINVAL;
      nttt::g_pack_persistent = (int)value;
      return NTTT_OK;
    case NTTT_TUNE_POOL_ORDER:
      if (value < 0 || value > 1) return NTTT_EINVAL;
      ctx->pool_order = value != 0;
      return NTTT_OK;
    case NTTT_TUNE_UPSAMPLE_STAGE_BYTES:
      if (value < 0 || value > 160 * 1024) return NTTT_EINVAL;
      ctx->upsample_stage_floats = (int)(value / 4);
      return NTTT_OK;
    default:
      return NTTT_EINVAL;
  }
}

int nttt_ctx_profile(nttt_ctx* ctx, int enable) {
  if (!ctx) return NTTT_EINVAL;
  if (enable)
    for (int i = 0; i <= kNumStages; ++i)
      if (!ctx->ev[i]) NTTT_CUDA(cudaEventCreate(&ctx->ev[i]));
  ctx->profile = enable != 0;
  ctx->n_ev = 0;
  return NTTT_OK;
}

int nttt_ctx_profile_read(nttt_ctx* ctx, float* ms_host, int capacity) {
  if (!ctx || !ms_host || capacity < kNumStages) return NTTT_EINVAL;
  if (ctx->n_ev != kNumStages + 1) return NTTT_EINVAL;  // no complete image recorded
  NTTT_CUDA(cudaEventSynchronize(ctx->ev[kNumStages]));
  for (int i = 0; i < kNumStages; ++i) NTTT_CUDA(cudaEventElapsedTime(&ms_host[i], ctx->ev[i], ctx->ev[i + 1]));
  return kNumStages;
}

const char* nttt_error_string(int code) {
  switch (code) {
    case NTTT_OK: return "ok";
    case NTTT_EINVAL: return "invalid argument";
    case NTTT_ENODEVICE: return "no CUDA device";
    case NTTT_ECUDA: return "CUDA error";
    case NTTT_EWORKSPACE: return "workspace too small";
    case NTTT_EUNSUPPORTED: return "unsupported shape";
    default: return "unknown error";
  }
}

const char* nttt_last_cuda_error(void) { return g_cuda_err; }

int nttt_ctx_create(nttt_ctx** out, int device) {
  if (!out) return NTTT_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    if (e != cudaSuccess) cuda_fail(e, "cudaGetDeviceCount");
    return NTTT_ENODEVICE;
  }
  if (device < 0 || device >= count) return NTTT_EINVAL;
  cudaDeviceProp prop;
  NTTT_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "device %d is sm_%d%d; libnttt_b200 is built for sm_100a only", device,
             prop.major, prop.minor);
    return NTTT_ENODEVICE;
  }
  NTTT_CUDA(cudaSetDevice(device));
  nttt_ctx* ctx = new nttt_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
#ifdef NTTT_ABLATE
  if (const char* e = getenv("NTTT_STOP_AFTER")) ctx->stop_after = atoi(e);
#endif
  *out = ctx;
  return NTTT_OK;
}

void nttt_ctx_destroy(nttt_ctx* ctx) {
  if (!ctx) return;
  if (ctx->side) cudaStreamDestroy(ctx->side);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  for (int i = 0; i < ctx->n_tables; ++i) free_axis_table(ctx->tables[i]);
  for (int i = 0; i < ctx->n_retired; ++i) free_axis_table(ctx->retired[i]);
  for (int i = 0; i < ctx->n_atlases; ++i) cudaFree(ctx->atlases[i].slab);
  if (ctx->scratch) cudaFree(ctx->scratch);
  for (int i = 0; i <= nttt_ctx::kMaxStages; ++i)
    if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  delete ctx;
}

int nttt_threshold_pack(const float* logits, int n, int h, int w, float thr, float off, uint32_t* bits, int32_t* area,
                        int32_t* box, int32_t* stab, int32_t* flags, void* stream) {
  if (n < 0 || h <= 0 || w <= 0) return NTTT_EINVAL;
  if (n > 0 && (!logits || !bits || !area || !box || !flags)) return NTTT_EINVAL;  // stab may be NULL
  return launch_lowres_pack(logits, n, h, w, thr, off, bits, area, box, stab, flags, nullptr, 0.0f, nullptr,
                            (cudaStream_t)stream);
}

int nttt_threshold_pack_stability(const float* logits, int n, int h, int w, float thr, float off, uint32_t* bits,
                                  int32_t* area, int32_t* box, int32_t* stab, float* stab_score, int32_t* flags,
                                  void* stream) {
  if (n < 0 || h <= 0 || w <= 0) return NTTT_EINVAL;
  if (n > 0 && (!logits || !bits || !area || !box || !stab || !stab_score || !flags)) return NTTT_EINVAL;
  return launch_lowres_pack(logits, n, h, w, thr, off, bits, area, box, stab, flags, nullptr, 0.0f, nullptr,
                            (cudaStream_t)stream, stab_score);
}

// host-side check + by-value table of the decoder's per-batch tensors
static int make_chunk_table(const float* const* chunks_host, int n_chunks, int chunk_prompts, int n, ChunkTable* out) {
  if (!chunks_host || n_chunks <= 0 || chunk_prompts <= 0) return NTTT_EINVAL;
  if (n_chunks > kMaxChunks) return NTTT_EUNSUPPORTED;
  if ((long long)n_chunks * chunk_prompts < n) return NTTT_EINVAL;
  for (int i = 0; i < kMaxChunks; ++i) out->base[i] = nullptr;
  for (int i = 0; i < n_chunks; ++i) {
    if (!chunks_host[i] || (reinterpret_cast<uintptr_t>(chunks_host[i]) & 15) != 0) return NTTT_EINVAL;
    out->base[i] = chunks_host[i];
  }
  return NTTT_OK;
}

int nttt_select_multimask(const float* ious, int n, int m, int first, const float* const* chunks_host, int n_chunks,
                          int chunk_prompts, int h, int w, const float** mask_ptr, float* score, void* stream) {
  if (n < 0 || m <= 0 || first < 0 || first >= m || h <= 0 || w <= 0) return NTTT_EINVAL;
  if (n == 0) return NTTT_OK;
  if (!ious || !mask_ptr || !score || ((size_t)h * w) % 4 != 0) return NTTT_EINVAL;
  ChunkTable t;
  int err = make_chunk_table(chunks_host, n_chunks, chunk_prompts, n, &t);
  if (err) return err;
  return launch_multimask_select(ious, n, m, first, t, chunk_prompts, (size_t)h * w, mask_ptr, score,
                                 (cudaStream_t)stream);
}

int nttt_threshold_pack_ptrs(const float* const* mask_ptr, const float* gate, float gate_min, int n, int h, int w,
                             float thr, float off, uint32_t* bits, int32_t* area, int32_t* box, int32_t* stab,
                             int32_t* flags, void* stream) {
  if (n < 0 || h <= 0 || w <= 0) return NTTT_EINVAL;
  if (n > 0 && (!mask_ptr || !bits || !area || !box || !flags)) return NTTT_EINVAL;
  return launch_lowres_pack(nullptr, n, h, w, thr, off, bits, area, box, stab, flags, gate, gate_min, mask_ptr,
                            (cudaStream_t)stream);
}

int nttt_project_masks(nttt_ctx* ctx, const uint32_t* bits, const int32_t* box, int n, int h, int w, int eh, int ew,
                       float* proj, void* stream) {
  if (!ctx || n < 0 || h <= 0 || w <= 0 || eh <= 0 || ew <= 0) return NTTT_EINVAL;
  if (n > 0 && (!bits || !box || !proj)) return NTTT_EINVAL;
  if (!projection_supported(ew, w) || !projection_supported(eh, h)) return NTTT_EUNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  ++ctx->epoch;
  AxisTable tx, ty;
  int err = ctx->axis(ew, w, s, &tx);
  if (err) return err;
  err = ctx->axis(eh, h, s, &ty);
  if (err) return err;
  return launch_project_masks(tx, ty, bits, box, n, h, w, eh, ew, proj, eh * ew, false, s);
}

size_t nttt_pool_workspace_bytes(int n, int e, int c) {
  const size_t ep = pad64(e);
  return align_up(sizeof(float) * (size_t)kPoolSplitsMax * n * c, 256) + align_up(2 * (size_t)n * 3 * ep, 256) +
         align_up(2 * (size_t)c * 3 * ep, 256);
}

int nttt_pool_normalize(nttt_ctx* ctx, const float* proj, const float* feat, const int32_t* area, int n, int e, int c,
                        float* obj_feats, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx || n < 0 || e <= 0 || c <= 0) return NTTT_EINVAL;
  if (n == 0) return NTTT_OK;
  if (!proj || !feat || !area || !obj_feats || !workspace) return NTTT_EINVAL;
  if (workspace_bytes < nttt_pool_workspace_bytes(n, e, c)) return NTTT_EWORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = static_cast<char*>(workspace);
  float* sums = reinterpret_cast<float*>(ws);
  char* a_split = ws + align_up(sizeof(float) * (size_t)kPoolSplitsMax * n * c, 256);
  char* b_split = a_split + align_up(2 * (size_t)n * 3 * pad64(e), 256);
  int n_partials = 1;
  int err = pool_contract(proj, feat, n, e, c, sums, a_split, b_split, &n_partials, s);
  if (err) return err;
  bool split_done;
  return normalize_rows(sums, n_partials, area, n, c, obj_feats, nullptr, &split_done, false, s);
}

int nttt_proto_prepare(const float* feats_ins_avg, int n_cls, int shots, int c, float* proto, void* stream) {
  if (n_cls <= 0 || shots <= 0 || c <= 0 || !feats_ins_avg || !proto) return NTTT_EINVAL;
  return launch_proto_prepare(feats_ins_avg, n_cls, shots, c, proto, (cudaStream_t)stream);
}

size_t nttt_similarity_workspace_bytes(int n, int c, int n_cls) {
  const size_t cp = pad64(c);
  return align_up(sizeof(float) * sim_partial_floats(n, n_cls, c), 256) + align_up(2 * (size_t)n * 3 * cp, 256) +
         align_up(2 * (size_t)n_cls * 3 * cp, 256);
}

int nttt_similarity_top1(nttt_ctx* ctx, const float* obj_feats, const float* proto, int n, int c, int n_cls,
                         float* sim, float* top_score, int32_t* top_label, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (!ctx || n < 0 || c <= 0 || n_cls <= 0) return NTTT_EINVAL;
  if (n == 0) return NTTT_OK;
  if (!obj_feats || !proto || !top_score || !top_label) return NTTT_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  if (!workspace || workspace_bytes < nttt_similarity_workspace_bytes(n, c, n_cls)) return NTTT_EWORKSPACE;
  char* ws = static_cast<char*>(workspace);
  float* partials = reinterpret_cast<float*>(ws);
  char* a_split = ws + align_up(sizeof(float) * sim_partial_floats(n, n_cls, c), 256);
  char* b_split = a_split + align_up(2 * (size_t)n * 3 * pad64(c), 256);
  return sim_top1(obj_feats, proto, nullptr, 0, 1.0f, n, c, n_cls, sim, partials, nullptr, top_score, top_label, a_split,
                  b_split, false, ctx->sm_count, s);
}

size_t nttt_similarity_neg_workspace_bytes(int n, int c, int n_cls, int l_neg) {
  const size_t cp = pad64(c);
  const size_t cols = (size_t)n_cls * l_neg;
  return align_up(sizeof(float) * sim_partial_floats(n, n_cls, c), 256) +
         align_up(sizeof(float) * sim_partial_floats(n, (int)cols, c), 256) + align_up(2 * (size_t)n * 3 * cp, 256) +
         align_up(2 * cols * 3 * cp, 256);
}

int nttt_similarity_neg_top1(nttt_ctx* ctx, const float* obj_feats, const float* proto_pos, const float* proto_neg,
                             int n, int c, int n_cls, int l_neg, float sigma, float* sim, float* top_score,
                             int32_t* top_label, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx || n < 0 || c <= 0 || n_cls <= 0 || l_neg <= 0 || !(sigma > 0.0f)) return NTTT_EINVAL;
  if (n == 0) return NTTT_OK;
  if (!obj_feats || !proto_pos || !proto_neg || !top_score || !top_label) return NTTT_EINVAL;
  if (!workspace || workspace_bytes < nttt_similarity_neg_workspace_bytes(n, c, n_cls, l_neg)) return NTTT_EWORKSPACE;
  char* ws = static_cast<char*>(workspace);
  float* partials = reinterpret_cast<float*>(ws);
  float* partials_neg = reinterpret_cast<float*>(ws + align_up(sizeof(float) * sim_partial_floats(n, n_cls, c), 256));
  char* a_split = reinterpret_cast<char*>(partials_neg) +
                  align_up(sizeof(float) * sim_partial_floats(n, n_cls * l_neg, c), 256);
  char* b_split = a_split + align_up(2 * (size_t)n * 3 * pad64(c), 256);
  return sim_top1(obj_feats, proto_pos, proto_neg, l_neg, sigma, n, c, n_cls, sim, partials, partials_neg, top_score,
                  top_label, a_split, b_split, false, ctx->sm_count, (cudaStream_t)stream);
}

size_t nttt_nms_workspace_bytes(int n) { return nms_workspace_bytes(n > 0 ? n : 1); }

int nttt_box_nms(const int32_t* box, const float* nms_scores, const int32_t* labels, const float* top_score, int n,
                 float iou_thr, int max_keep, int32_t* keep, int32_t* n_keep, int32_t* sel, int32_t* n_sel,
                 void* workspace, size_t workspace_bytes, void* stream) {
  if (n < 0 || !keep || !n_keep || !sel || !n_sel) return NTTT_EINVAL;
  if (n > 0 && (!box || !nms_scores || !labels || !top_score || !workspace)) return NTTT_EINVAL;
  return launch_box_nms(box, nms_scores, labels, top_score, n, iou_thr, max_keep, keep, n_keep, sel, n_sel, workspace,
                        workspace_bytes, 0.0f, 0, (cudaStream_t)stream);
}

// scratch for the cross-CTA per-mask statistics of the stand-alone resize entry is owned by the ctx
static int ensure_scratch(nttt_ctx* ctx, int max_sel, int oh, int ow, int32_t** out) {
  const size_t need = upsample_scratch_bytes(max_sel, oh, ow);
  if (need > ctx->scratch_cap) {
    if (ctx->scratch) {
      NTTT_CUDA(cudaDeviceSynchronize());  // kernels of earlier calls may still use it (rare: the need only grows)
      cudaFree(ctx->scratch);
    }
    ctx->scratch = nullptr;
    ctx->scratch_cap = 0;
    NTTT_CUDA(cudaMalloc(&ctx->scratch, need));
    ctx->scratch_cap = need;
  }
  *out = ctx->scratch;
  return NTTT_OK;
}

static int upsample_entry(nttt_ctx* ctx, const float* logits, const float* const* mask_ptr, const uint32_t* bits_lr,
                          const int32_t* box_lr, const int32_t* flags_lr, int ih, int iw, const int32_t* sel,
                          const int32_t* n_sel, int max_sel, int oh, int ow, uint32_t* bits_full, int32_t* rect,
                          int32_t* area_full, int32_t* box_full, void* stream) {
  if (!ctx || max_sel < 0 || ih <= 0 || iw <= 0 || oh <= 0 || ow <= 0) return NTTT_EINVAL;
  if (max_sel == 0) return NTTT_OK;
  if ((!logits && !mask_ptr) || !bits_lr || !box_lr || !flags_lr || !sel || !n_sel || !bits_full || !rect || !area_full ||
      !box_full)
    return NTTT_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  ++ctx->epoch;
  AxisTable tx, ty;
  int err = ctx->axis(iw, ow, s, &tx);
  if (err) return err;
  err = ctx->axis(ih, oh, s, &ty);
  if (err) return err;
  int32_t* scratch = nullptr;
  err = ensure_scratch(ctx, max_sel, oh, ow, &scratch);
  if (err) return err;
  return launch_upsample_pack(tx, ty, logits, bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, oh, ow,
                              bits_full, rect, area_full, box_full, scratch, mask_ptr, s, ctx->upsample_stage_floats,
                              ctx->sm_count);
}

int nttt_upsample_threshold_pack(nttt_ctx* ctx, const float* logits, const uint32_t* bits_lr, const int32_t* box_lr,
                                 const int32_t* flags_lr, int ih, int iw, const int32_t* sel, const int32_t* n_sel,
                                 int max_sel, int oh, int ow, uint32_t* bits_full, int32_t* rect, int32_t* area_full,
                                 int32_t* box_full, void* stream) {
  return upsample_entry(ctx, logits, nullptr, bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, oh, ow, bits_full,
                        rect, area_full, box_full, stream);
}

int nttt_upsample_threshold_pack_ptrs(nttt_ctx* ctx, const float* const* mask_ptr, const uint32_t* bits_lr,
                                      const int32_t* box_lr, const int32_t* flags_lr, int ih, int iw, const int32_t* sel,
                                      const int32_t* n_sel, int max_sel, int oh, int ow, uint32_t* bits_full,
                                      int32_t* rect, int32_t* area_full, int32_t* box_full, void* stream) {
  return upsample_entry(ctx, nullptr, mask_ptr, bits_lr, box_lr, flags_lr, ih, iw, sel, n_sel, max_sel, oh, ow, bits_full,
                        rect, area_full, box_full, stream);
}

size_t nttt_mask_ios_workspace_bytes(int max_sel) { return ios_workspace_bytes(max_sel > 0 ? max_sel : 1); }

int nttt_mask_ios(const uint32_t* bits_full, const int32_t* rect, const int32_t* area_full, const int32_t* box_full,
                  const int32_t* sel, const int32_t* n_sel, int max_sel, int oh, int ow, const int32_t* labels,
                  const float* obj_feats, int c, float* ios, int32_t* inter_out, void* workspace,
                  size_t workspace_bytes, void* stream) {
  if (max_sel < 0 || oh <= 0 || ow <= 0 || c <= 0) return NTTT_EINVAL;
  if (max_sel == 0) return NTTT_OK;
  if (!bits_full || !rect || !area_full || !box_full || !sel || !n_sel || !labels || !obj_feats || !ios)
    return NTTT_EINVAL;
  if (!workspace || workspace_bytes < ios_workspace_bytes(max_sel)) return NTTT_EWORKSPACE;
  return launch_mask_ios(bits_full, rect, area_full, box_full, sel, n_sel, max_sel, oh, ow, labels, obj_feats, c, ios,
                         inter_out, workspace, true, (cudaStream_t)stream);
}

int nttt_decay_topk(const float* top_score, const int32_t* labels, const float* ios, const int32_t* sel,
                    const int32_t* n_sel, int max_sel, int num_out, const uint32_t* bits_full, const int32_t* rect,
                    const int32_t* box_full, int oh, int ow, uint8_t* out_masks, int64_t* out_boxes, float* out_scores,
                    int64_t* out_labels, int32_t* out_index, int32_t* out_slot, int32_t* n_out, void* stream) {
  if (max_sel < 0 || num_out < 0 || oh <= 0 || ow <= 0) return NTTT_EINVAL;
  if (!n_out) return NTTT_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  if (max_sel == 0 || num_out == 0) {
    NTTT_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int32_t), s));
    return NTTT_OK;
  }
  if (!top_score || !labels || !ios || !sel || !n_sel || !bits_full || !rect || !box_full || !out_masks || !out_boxes ||
      !out_scores || !out_labels || !out_index || !out_slot)
    return NTTT_EINVAL;
  int err = launch_decay_rank(top_score, labels, ios, sel, n_sel, max_sel, num_out, box_full, nullptr, out_boxes, out_scores,
                              out_labels, out_index, out_slot, n_out, nullptr, s);
  if (err) return err;
  return launch_unpack(bits_full, rect, out_slot, n_out, num_out, oh, ow, out_masks, s);
}

int nttt_unpack_masks(const uint32_t* bits_full, const int32_t* rect, const int32_t* n_sel, int max_sel, int oh, int ow,
                      uint8_t* masks_u8, void* stream) {
  if (max_sel < 0 || oh <= 0 || ow <= 0) return NTTT_EINVAL;
  if (max_sel == 0) return NTTT_OK;
  if (!bits_full || !rect || !n_sel || !masks_u8) return NTTT_EINVAL;
  return launch_unpack(bits_full, rect, nullptr, n_sel, max_sel, oh, ow, masks_u8, (cudaStream_t)stream);
}

int nttt_rle_encode(const uint32_t* bits_full, const int32_t* rect, const int32_t* slot, const int32_t* count,
                    int max_count, int oh, int ow, int cap_counts, int cap_chars, uint32_t* counts, int32_t* n_counts,
                    uint8_t* chars, int32_t* n_chars, void* stream) {
  if (max_count < 0 || oh <= 0 || ow <= 0 || cap_counts <= 0 || cap_chars <= 0) return NTTT_EINVAL;
  if (max_count == 0) return NTTT_OK;
  if (!bits_full || !rect || !count || !counts || !n_counts || !chars || !n_chars) return NTTT_EINVAL;
  return launch_rle_encode(bits_full, rect, slot, count, max_count, oh, ow, cap_counts, cap_chars, counts, n_counts, chars,
                           n_chars, (cudaStream_t)stream);
}

int nttt_rle_compact(const uint8_t* chars, const int32_t* n_chars, int n_masks, int cap_chars, uint8_t* out,
                     int64_t out_cap, void* stream) {
  if (n_masks < 0 || cap_chars <= 0 || out_cap < 0) return NTTT_EINVAL;
  if (n_masks == 0) return NTTT_OK;
  if (!chars || !n_chars || !out) return NTTT_EINVAL;
  return launch_rle_compact(chars, n_chars, n_masks, cap_chars, out, (long long)out_cap, (cudaStream_t)stream);
}

int nttt_fill_pool_accumulate(const float* feat, const float* soft_mask, int mh, int mw, int eh, int ew, int c,
                              float* sum_slot, float* wsum_slot, float* mask_lowres_out, void* stream) {
  if (!feat || !soft_mask || !sum_slot || !wsum_slot || mh <= 0 || mw <= 0 || eh <= 0 || ew <= 0 || c <= 0)
    return NTTT_EINVAL;
  return launch_fill_pool(feat, soft_mask, 1, mh, mw, eh, ew, c, sum_slot, wsum_slot, mask_lowres_out, 1,
                          (cudaStream_t)stream);
}

int nttt_fill_pool_batch(const float* feat, const float* soft_mask, int b, int mh, int mw, int eh, int ew, int c,
                         float* sums, float* wsums, float* masks_lowres, void* stream) {
  if (b < 0 || mh <= 0 || mw <= 0 || eh <= 0 || ew <= 0 || c <= 0) return NTTT_EINVAL;
  if (b == 0) return NTTT_OK;
  if (!feat || !soft_mask || !sums || !wsums) return NTTT_EINVAL;
  return launch_fill_pool(feat, soft_mask, b, mh, mw, eh, ew, c, sums, wsums, masks_lowres, 0, (cudaStream_t)stream);
}

int nttt_fill_scatter(const float* sums, const float* wsums, const float* masks_lowres, const int32_t* slot, int n, int c,
                      int e, float* feats_sum, float* mask_sum, float* masks, void* stream) {
  if (n < 0 || c <= 0 || e <= 0) return NTTT_EINVAL;
  if (n == 0) return NTTT_OK;
  if (!sums || !wsums || !slot || !feats_sum || !mask_sum) return NTTT_EINVAL;
  if ((masks == nullptr) != (masks_lowres == nullptr)) return NTTT_EINVAL;
  return launch_fill_scatter(sums, wsums, masks_lowres, slot, n, c, e, feats_sum, mask_sum, masks, (cudaStream_t)stream);
}

int nttt_fill_finalize(const float* sum, const float* wsum, int n_cls, int shots, int c, float* feats_ins_avg,
                       float* feats_avg, void* stream) {
  if (!sum || !wsum || !feats_ins_avg || !feats_avg || n_cls <= 0 || shots <= 0 || c <= 0) return NTTT_EINVAL;
  return launch_fill_finalize(sum, wsum, n_cls, shots, c, feats_ins_avg, feats_avg, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------
// whole-image pipeline
// ---------------------------------------------------------------------------------------------------
struct MatchLayout {
  uint32_t* bits_lr; int32_t* area_lr; int32_t* box_lr; int32_t* stab; int32_t* flags;
  float* proj; float* sums; float* obj_feats; float* sim; float* sim_part; float* sim_part_neg; float* top_score; int32_t* top_label;
  char* a_split; char* b_split; char* p_split;
  int32_t* pool_perm; uint32_t* pool_active; uint8_t* b_nonfinite;
  void* nms_ws; size_t nms_ws_bytes; int32_t* keep; int32_t* sel;
  uint32_t* bits_full; uint32_t* bits_t; int32_t* rect; int32_t* area_full; int32_t* box_full; int32_t* scratch;
  float* ios; void* ios_ws; int32_t* out_slot;
  const float** mask_ptr; float* plane_score;
  size_t total;
};

static MatchLayout carve(void* ws, int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int oh, int ow,
                         int max_sel, int num_out, int l_neg) {
  Carver cv(ws);
  MatchLayout L;
  const size_t p = (size_t)lr_h * lr_w;
  L.bits_lr = cv.take<uint32_t>((size_t)n * (p / 32));
  L.area_lr = cv.take<int32_t>(n);
  L.box_lr = cv.take<int32_t>((size_t)n * 4);
  L.stab = cv.take<int32_t>((size_t)n * 2);
  L.flags = cv.take<int32_t>(n);
  L.proj = cv.take<float>((size_t)n * eh * ew);
  L.sums = cv.take<float>((size_t)kPoolSplitsMax * n * c);
  L.obj_feats = cv.take<float>((size_t)n * c);
  L.sim = cv.take<float>((size_t)n * n_cls);
  L.sim_part = cv.take<float>(sim_partial_floats(n, n_cls, c));
  L.sim_part_neg = cv.take<float>(l_neg > 0 ? sim_partial_floats(n, n_cls * l_neg, c) : 1);
  {
    const size_t kmax = (size_t)3 * (pad64(eh * ew) > pad64(c) ? pad64(eh * ew) : pad64(c));
    size_t rows_b = (size_t)(c > n_cls ? c : n_cls);
    if ((size_t)n_cls * (l_neg > 0 ? l_neg : 0) > rows_b) rows_b = (size_t)n_cls * l_neg;
    L.a_split = cv.take<char>(2 * (size_t)n * kmax);
    L.b_split = cv.take<char>(2 * rows_b * kmax);
    L.p_split = cv.take<char>(2 * (size_t)n_cls * 3 * pad64(c));  // split prototypes (prepared off the critical path)
    L.pool_perm = cv.take<int32_t>(n > 0 ? n : 1);       // spatial row order of the pooling GEMM (pool_order_kernel)
    L.pool_active = cv.take<uint32_t>(n > 0 ? n : 1);    // per operand row: its non-zero k-blocks
    L.b_nonfinite = cv.take<uint8_t>((size_t)(pad64(eh * ew) / 64) * ((c + 31) / 32));
  }
  L.top_score = cv.take<float>(n);
  L.top_label = cv.take<int32_t>(n);
  L.nms_ws_bytes = nms_workspace_bytes(n > 0 ? n : 1);
  L.nms_ws = cv.take<char>(L.nms_ws_bytes);
  L.keep = cv.take<int32_t>(max_sel > 0 ? max_sel : 1);
  L.sel = cv.take<int32_t>(max_sel > 0 ? max_sel : 1);
  L.bits_full = cv.take<uint32_t>((size_t)max_sel * oh * ((ow + 31) / 32));
  L.bits_t = cv.take<uint32_t>((size_t)max_sel * oh * ((ow + 31) / 32));  // word-column-major copy for mask_ios
  L.rect = cv.take<int32_t>((size_t)max_sel * 4);
  L.area_full = cv.take<int32_t>(max_sel > 0 ? max_sel : 1);
  L.box_full = cv.take<int32_t>((size_t)max_sel * 4);
  L.scratch = cv.take<int32_t>(upsample_scratch_bytes(max_sel > 0 ? max_sel : 1, oh, ow) / sizeof(int32_t) + 1);
  L.ios = cv.take<float>(max_sel > 0 ? max_sel : 1);
  L.ios_ws = cv.take<char>(ios_workspace_bytes(max_sel > 0 ? max_sel : 1));
  L.out_slot = cv.take<int32_t>(num_out > 0 ? num_out : 1);
  L.mask_ptr = cv.take<const float*>(n > 0 ? n : 1);
  L.plane_score = cv.take<float>(n > 0 ? n : 1);
  L.total = align_up(cv.off, 256);
  return L;
}

size_t nttt_match_workspace_bytes(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h, int ori_w,
                                  int max_sel) {
  if (n < 0 || lr_h <= 0 || lr_w <= 0 || eh <= 0 || ew <= 0 || c <= 0 || n_cls <= 0 || ori_h <= 0 || ori_w <= 0 ||
      max_sel < 0)
    return 0;
  return carve(nullptr, n, lr_h, lr_w, eh, ew, c, n_cls, ori_h, ori_w, max_sel, max_sel, 0).total;
}

size_t nttt_match_workspace_bytes_neg(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h, int ori_w,
                                      int max_sel, int l_neg) {
  if (n < 0 || lr_h <= 0 || lr_w <= 0 || eh <= 0 || ew <= 0 || c <= 0 || n_cls <= 0 || ori_h <= 0 || ori_w <= 0 ||
      max_sel < 0 || l_neg < 0)
    return 0;
  return carve(nullptr, n, lr_h, lr_w, eh, ew, c, n_cls, ori_h, ori_w, max_sel, max_sel, l_neg).total;
}

size_t nttt_match_workspace_bytes_sized(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h, int ori_w,
                                        int max_sel, int l_neg, int min_h, int min_w) {
  if (min_h <= 0 || min_w <= 0 || min_h > ori_h || min_w > ori_w) return 0;
  // (every buffer of the workspace grows with the output size: the capacity's layout serves the whole range)
  return nttt_match_workspace_bytes_neg(n, lr_h, lr_w, eh, ew, c, n_cls, ori_h, ori_w, max_sel, l_neg);
}

int nttt_ctx_atlas_stats(nttt_ctx* ctx, size_t* bytes_host, double* build_ms_host) {
  if (!ctx) return NTTT_EINVAL;
  size_t bytes = 0;
  double ms = 0.0;
  for (int i = 0; i < ctx->n_atlases; ++i) {
    bytes += ctx->atlases[i].bytes;
    ms += ctx->atlases[i].build_ms;
  }
  if (bytes_host) *bytes_host = bytes;
  if (build_ms_host) *build_ms_host = ms;
  return ctx->n_atlases;
}

// range == nullptr: nttt_match_image (the size is a->ori_h x a->ori_w); otherwise nttt_match_image_sized
// in_dev != nullptr: nttt_match_image_bound (the input pointers of `a` are ignored; the kernels that read the inputs
// take their addresses from *in_dev)
static int match_impl(nttt_ctx* ctx, const nttt_match_args* a, const nttt_match_size_range* range, void* stream,
                      const nttt_match_inputs* in_dev = nullptr) {
  if (!ctx || !a) return NTTT_EINVAL;
  if (a->n < 0 || a->lr_h <= 0 || a->lr_w <= 0 || a->eh <= 0 || a->ew <= 0 || a->c <= 0 || a->n_cls <= 0 ||
      a->ori_h <= 0 || a->ori_w <= 0 || a->num_out_instance < 0 || a->max_sel < 0)
    return NTTT_EINVAL;
  if (range && (!range->ori_hw_dev || range->min_h <= 0 || range->min_w <= 0 || range->min_h > a->ori_h ||
                range->min_w > a->ori_w))
    return NTTT_EINVAL;
  if (range && (a->ori_h >= 65536 || a->ori_w >= 65536)) return NTTT_EUNSUPPORTED;
  if (!a->counts || !a->workspace) return NTTT_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  const int n = a->n, max_sel = a->max_sel, num_out = a->num_out_instance;
  if (n == 0 || max_sel == 0) {
    NTTT_CUDA(cudaMemsetAsync(a->counts, 0, 4 * sizeof(int32_t), s));
    return NTTT_OK;
  }
  const bool multi = a->n_multi > 1;
  const bool bound = in_dev != nullptr;
  const bool chunked = multi && (bound ? a->n_chunks > 0 : a->logits_chunks_host != nullptr);
  const bool want_rle = a->rle_chars != nullptr;
  if ((!bound && ((!a->logits && !chunked) || (!multi && !a->pred_ious) || !a->tar_feat)) || !a->proto ||
      (!a->out_masks && !want_rle) || !a->out_boxes || !a->out_scores || !a->out_labels || !a->out_index)
    return NTTT_EINVAL;
  if (bound && chunked &&
      (a->n_chunks > kMaxChunks || a->chunk_prompts <= 0 || (long long)a->n_chunks * a->chunk_prompts < n))
    return NTTT_EINVAL;
  if (want_rle && (!a->rle_counts || !a->rle_n_counts || !a->rle_n_chars || a->rle_cap_counts <= 0 || a->rle_cap_chars <= 0))
    return NTTT_EINVAL;
  if (multi && ((!bound && !a->multi_ious) || a->multi_first < 0 || a->multi_first >= a->n_multi)) return NTTT_EINVAL;
  const int l_neg = a->proto_neg ? a->l_neg : 0;
  if (a->proto_neg && (a->l_neg <= 0 || !(a->sigma > 0.0f))) return NTTT_EINVAL;
  MatchLayout L = carve(a->workspace, n, a->lr_h, a->lr_w, a->eh, a->ew, a->c, a->n_cls, a->ori_h, a->ori_w, max_sel,
                        num_out, l_neg);
  if (a->workspace_bytes < L.total) return NTTT_EWORKSPACE;
  if (!projection_supported(a->ew, a->lr_w) || !projection_supported(a->eh, a->lr_h)) return NTTT_EUNSUPPORTED;
  float* obj_feats = a->obj_feats ? a->obj_feats : L.obj_feats;
  float* sim = a->sim ? a->sim : L.sim;
  int32_t* sel = a->sel ? a->sel : L.sel;
  float* ios = a->ios ? a->ios : L.ios;
  struct LaunchMode {  // the launch shapes of this call (common.cuh: t_low_latency), restored on every return path
    bool prev;
    explicit LaunchMode(bool v) : prev(nttt::t_low_latency) { nttt::t_low_latency = v; }
    ~LaunchMode() { nttt::t_low_latency = prev; }
  } launch_mode(a->low_latency != 0);
  ++ctx->epoch;
  AxisTable px, py, ux, uy;
  int err = ctx->axis(a->ew, a->lr_w, s, &px);
  if (err) return err;
  if ((err = ctx->axis(a->eh, a->lr_h, s, &py))) return err;
  // sized: the resize tables of every size of the range, and what the kernels read the size from
  const SizedAtlas* atlas = nullptr;
  SizedDims sd{};
  if (range) {
    if ((err = ctx->sized_atlas(a->lr_h, a->lr_w, range->min_h, range->min_w, a->ori_h, a->ori_w, s, &atlas))) return err;
    sd = SizedDims{range->ori_hw_dev, atlas->ay, atlas->ax, a->counts, range->min_h, range->min_w, a->ori_h, a->ori_w};
  } else {
    if ((err = ctx->axis(a->lr_w, a->ori_w, s, &ux))) return err;
    if ((err = ctx->axis(a->lr_h, a->ori_h, s, &uy))) return err;
  }
  const SizedDims* sized = range ? &sd : nullptr;
  const int e = a->eh * a->ew;

  ctx->n_ev = 0;
#define NTTT_MARK()                                                              \
  do {                                                                           \
    if (ctx->profile) { NTTT_CUDA(cudaEventRecord(ctx->ev[ctx->n_ev], s)); ++ctx->n_ev; } \
  } while (0)
  // Ablation builds only (-DNTTT_ABLATE, `NTTT_BUILD_ABLATE=1 python build.py`): NTTT_STOP_AFTER=<k>, read once at
  // ctx creation, ends the pipeline after its k-th stage so that tools/ablate.py can measure the marginal cost of each
  // stage with several images in flight.  The product library does not contain this switch.
#ifdef NTTT_ABLATE
  int stage_no = 0;
#define NTTT_STOP_CHECK() if (ctx->stop_after > 0 && ++stage_no >= ctx->stop_after) return NTTT_OK
#else
#define NTTT_STOP_CHECK() (void)0
#endif
#define NTTT_STEP_QUIET(call) \
  do {                        \
    err = (call);             \
    if (err) return err;      \
  } while (0)
#define NTTT_STEP(call)                                        \
  do {                                                         \
    err = (call);                                              \
    if (err) return err;                                       \
    NTTT_MARK();                                               \
    NTTT_STOP_CHECK();                                         \
  } while (0)
  // candidate selection (§8f rank 2): resolve the best decoder plane per prompt; its IoU is the score from here on
  const float* const* mask_ptr = nullptr;
  const float* pred_ious = a->pred_ious;
  // bound inputs: the logits are reached through mask_ptr only, and the features through feat_at
  const float* logits = bound ? nullptr : a->logits;
  const float* const* feat_at = bound ? &in_dev->tar_feat : nullptr;
  if (bound) {
    if (multi)
      err = launch_multimask_select(nullptr, n, a->n_multi, a->multi_first, ChunkTable{}, chunked ? a->chunk_prompts : n,
                                    (size_t)a->lr_h * a->lr_w, L.mask_ptr, L.plane_score, s, &in_dev->multi_ious,
                                    chunked ? in_dev->chunks : &in_dev->logits);
    else
      err = launch_plane_resolve(in_dev, n, (size_t)a->lr_h * a->lr_w, L.mask_ptr, L.plane_score, s);
    if (err) return err;
    mask_ptr = L.mask_ptr;
    pred_ious = L.plane_score;
  } else if (multi) {
    ChunkTable ct;
    const float* one = a->logits;
    err = chunked ? make_chunk_table(a->logits_chunks_host, a->n_chunks, a->chunk_prompts, n, &ct)
                  : make_chunk_table(&one, 1, n, n, &ct);
    if (err) return err;
    if ((err = launch_multimask_select(a->multi_ious, n, a->n_multi, a->multi_first, ct, chunked ? a->chunk_prompts : n,
                                       (size_t)a->lr_h * a->lr_w, L.mask_ptr, L.plane_score, s)))
      return err;
    mask_ptr = L.mask_ptr;
    pred_ious = L.plane_score;
  }
  NTTT_MARK();
  // low-latency mode: the two operand preparations that do not depend on the masks (features -> transposed split
  // operand, prototypes -> split operand) run on the context's side stream while the main stream reads the logits
  const bool forked = a->low_latency != 0 && ctx->side_ready();
  // Once the side stream's work is recorded in ev_join, every return makes `s` wait for it: an early return must neither
  // leave the side stream writing the workspace after the call nor leave a stream capture unjoined.
  struct SideJoin {
    cudaStream_t s;
    cudaEvent_t ev = nullptr;  // armed while not null
    ~SideJoin() { if (ev) cudaStreamWaitEvent(s, ev, 0); }
  } side_join{s};
  if (forked) {
    NTTT_CUDA(cudaEventRecord(ctx->ev_fork, s));
    NTTT_CUDA(cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0));
    err = launch_split_transpose(a->tar_feat, a->c, a->c, e, pad64(e), 1, L.b_split, ctx->side, nullptr, feat_at);
    if (err) return err;
    err = launch_split_rows(a->proto, a->c, a->n_cls, a->c, pad64(a->c), 1, L.p_split, ctx->side);
    if (err) return err;
    NTTT_CUDA(cudaEventRecord(ctx->ev_join, ctx->side));
    side_join.ev = ctx->ev_join;
  }
  // a6/a9/a15: one pass over the logits
  // (the stability counts of a15 are not read on this path, so the pipeline does not pay for them)
  NTTT_STEP(launch_lowres_pack(logits, n, a->lr_h, a->lr_w, 0.0f, 1.0f, L.bits_lr, L.area_lr, L.box_lr, nullptr,
                               L.flags, a->filter_iou ? pred_ious : nullptr, a->iou_thr, mask_ptr, s));
  // a6/a7: projection + pooling contraction + normalisation
  // Many images in flight: the pooling GEMM runs on spatially ordered rows and skips the k-blocks a tile of masks does
  // not touch (~45 % of them).  Needs the vector normalisation path (it undoes the order) and <= 32 k-blocks per segment.
  const bool ordered = !a->low_latency && ctx->pool_order && n > 128 && n <= 8192 && pad64(e) / 64 <= 32 &&
                       (a->c == 384 || a->c == 768 || a->c == 1024 || a->c == 1536);
  if (ordered) NTTT_STEP_QUIET(launch_pool_order(L.box_lr, n, a->lr_h, L.pool_perm, s));
  NTTT_STEP(launch_project_masks(px, py, L.bits_lr, L.box_lr, n, a->lr_h, a->lr_w, a->eh, a->ew, L.a_split, pad64(e),
                                 true, s, ordered ? L.pool_perm : nullptr, ordered ? L.pool_active : nullptr));
  int n_partials = 1;
  if (forked) {
    NTTT_CUDA(cudaStreamWaitEvent(s, ctx->ev_join, 0));
    side_join.ev = nullptr;
    nttt::t_chain_break = true;  // the pooling GEMM depends on the side stream as well: launched the ordinary way
  }
  NTTT_STEP(pool_contract(nullptr, a->tar_feat, n, e, a->c, L.sums, L.a_split, L.b_split, &n_partials, s,
                          a->low_latency != 0, forked, ordered ? L.pool_active : nullptr, L.b_nonfinite, feat_at));
  bool a_ready = false;
  NTTT_STEP(normalize_rows(L.sums, n_partials, L.area_lr, n, a->c, obj_feats, L.a_split, &a_ready,
                           a->proto_neg != nullptr, s, ordered ? L.pool_perm : nullptr));
  // a7/a8: similarity + top-1
  NTTT_STEP(sim_top1(obj_feats, a->proto, a->proto_neg, l_neg, a->sigma, n, a->c, a->n_cls, a->sim, L.sim_part,
                     L.sim_part_neg, L.top_score, L.top_label, L.a_split, L.b_split, a_ready, ctx->sm_count, s, L.p_split,
                     forked));
  // a10/a11
  NTTT_STEP(launch_box_nms(L.box_lr, pred_ious, L.top_label, L.top_score, n, a->nms_thr, max_sel, L.keep,
                           a->counts + 0, sel, a->counts + 1, L.nms_ws, L.nms_ws_bytes, a->iou_thr, a->filter_iou, s));
  // a12/a9 (sized: ux, uy are empty, the tables come from the atlas)
  bool wrote_t = false;  // the resize left the word-column-major copy of the packed masks instead of the row-major one
  NTTT_STEP(launch_upsample_pack(ux, uy, logits, L.bits_lr, L.box_lr, L.flags, a->lr_h, a->lr_w, sel, a->counts + 1,
                                 max_sel, a->ori_h, a->ori_w, L.bits_full, L.rect, L.area_full, L.box_full, L.scratch,
                                 mask_ptr, s, ctx->upsample_stage_floats, ctx->sm_count, L.bits_t, &wrote_t,
                                 a->low_latency != 0, ios_pair_counters(L.ios_ws, max_sel), sized, atlas));
  // the packed full-resolution masks from here on: word-column major when the resize wrote that layout, row-major otherwise
  const uint32_t* packed = wrote_t ? L.bits_t : L.bits_full;
  // a13
  NTTT_STEP(launch_mask_ios(L.bits_full, L.rect, L.area_full, L.box_full, sel, a->counts + 1, max_sel, a->ori_h,
                            a->ori_w, L.top_label, obj_feats, a->c, ios, a->ios_inter, L.ios_ws, false, s,
                            wrote_t ? L.bits_t : nullptr, /*counters_zeroed=*/wrote_t && a->low_latency != 0, sized));  // (folding the metadata
  // kernel into the pair kernel takes 1 us off a single image's chain and costs 0.3 us/image with images in flight)
  // a14
  NTTT_STEP(launch_decay_rank(L.top_score, L.top_label, ios, sel, a->counts + 1, max_sel, num_out, L.box_full,
                              L.area_full,
                              a->out_boxes, a->out_scores, a->out_labels, a->out_index, L.out_slot, a->counts + 2,
                              nullptr, s));
  if (!a->out_masks)
    NTTT_MARK();  // RLE-only output: the dense bool masks are never produced
  else if (a->out_prev_rect)
    NTTT_STEP(launch_unpack_sparse(packed, L.rect, L.out_slot, a->counts + 2, num_out, a->ori_h, a->ori_w,
                                   a->out_masks, a->out_prev_rect, s, wrote_t, sized));
  else
    NTTT_STEP(launch_unpack(packed, L.rect, L.out_slot, a->counts + 2, num_out, a->ori_h, a->ori_w, a->out_masks,
                            s, wrote_t, sized));
  // §8f rank 1: COCO RLE of the outputs straight from the packed words
  if (want_rle)
    NTTT_STEP(launch_rle_encode(packed, L.rect, L.out_slot, a->counts + 2, num_out, a->ori_h, a->ori_w,
                                a->rle_cap_counts, a->rle_cap_chars, a->rle_counts, a->rle_n_counts, a->rle_chars,
                                a->rle_n_chars, s, wrote_t, sized));
  else
    NTTT_MARK();
#undef NTTT_STEP
#undef NTTT_STOP_CHECK
#undef NTTT_MARK
  return NTTT_OK;
}

int nttt_match_image(nttt_ctx* ctx, const nttt_match_args* a, void* stream) { return match_impl(ctx, a, nullptr, stream); }

int nttt_match_image_sized(nttt_ctx* ctx, const nttt_match_args* a, const nttt_match_size_range* range, void* stream) {
  if (!range) return NTTT_EINVAL;
  return match_impl(ctx, a, range, stream);
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int nttt_match_bind(nttt_match_inputs* inputs_dev, const nttt_match_inputs* host, const nttt_match_args* shapes,
                    void* stream) {
  if (!inputs_dev || !host || !shapes || (reinterpret_cast<uintptr_t>(inputs_dev) & 7) != 0) return NTTT_EINVAL;
  if (shapes->n < 0 || !host->tar_feat) return NTTT_EINVAL;
  const int n = shapes->n;
  if (shapes->n_multi > 1) {
    if (!host->multi_ious) return NTTT_EINVAL;
    if (shapes->n_chunks > 0) {
      const int k = shapes->n_chunks;
      if (k > kMaxChunks || shapes->chunk_prompts <= 0 || (long long)k * shapes->chunk_prompts < n) return NTTT_EINVAL;
      for (int i = 0; i < k; ++i)
        if (!host->chunks[i] || !aligned16(host->chunks[i])) return NTTT_EINVAL;
    } else if (!host->logits || !aligned16(host->logits)) {
      return NTTT_EINVAL;
    }
  } else if (!host->logits || !aligned16(host->logits) || !host->pred_ious) {
    return NTTT_EINVAL;
  }
  return launch_match_bind(*host, inputs_dev, (cudaStream_t)stream);
}

int nttt_match_image_bound(nttt_ctx* ctx, const nttt_match_args* a, const nttt_match_size_range* range,
                           const nttt_match_inputs* inputs_dev, void* stream) {
  if (!inputs_dev) return NTTT_EINVAL;
  return match_impl(ctx, a, range, stream, inputs_dev);
}

}  // extern "C"
