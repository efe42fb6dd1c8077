/*
 * nttt_b200.h — C-ABI of libnttt_b200.so: the B200-native (sm_100a) reference-matching stage of
 * DogRog/no-time-to-train.
 *
 * The reference has no FFI: its seam is the Python class `Sam2MatchingBaselineNoAMG`
 * (no_time_to_train/models/Sam2MatchingBaseline_noAMG.py:128-765).  Each entry point below replaces the
 * library calls of one section of that class; the reference file:line it replaces is cited per function.
 * `no-time-to-train_b200/model.py` is the host-side mirror that binds these with ctypes (see
 * INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is DEVICE memory unless the name ends in `_host`;
 *   - the caller owns every buffer (inputs, outputs, workspace); nothing is allocated per call;
 *   - `stream` is a `cudaStream_t` passed as `void*`; every call is stream-ordered and never
 *     synchronises the device; data-dependent counts are returned in device memory;
 *   - return value: 0 on success, a negative `NTTT_E*` code otherwise (never throws);
 *   - there is no CPU path: on a machine without an sm_100 device the compute entries return
 *     NTTT_ENODEVICE / the CUDA launch error.
 *
 * Bit-packed masks: one `uint32_t` word holds 32 consecutive pixels of ONE row, bit b = pixel x0+b
 * (LSB first).  A row of W pixels occupies `words = (W+31)/32` words; pad bits are zero.
 */
#ifndef NTTT_B200_H
#define NTTT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NTTT_VERSION 200

enum {
  NTTT_OK = 0,
  NTTT_EINVAL = -1,     /* bad argument (null pointer, non-positive size, unsupported shape) */
  NTTT_ENODEVICE = -2,  /* no CUDA device / not an sm_100 device */
  NTTT_ECUDA = -3,      /* a CUDA runtime / driver call failed; see nttt_last_cuda_error() */
  NTTT_EWORKSPACE = -4, /* workspace too small */
  NTTT_EUNSUPPORTED = -5
};

typedef struct nttt_ctx nttt_ctx;

int nttt_version(void);
/* 1 if the library was built with -DNTTT_ABLATE (honours NTTT_STOP_AFTER for tools/ablate.py);
 * the product build returns 0 and does not contain the switch. */
int nttt_build_is_ablation(void);
const char* nttt_error_string(int code);
/* text of the last CUDA error seen by this thread's calls ("" if none) */
const char* nttt_last_cuda_error(void);

/* Per-device context: caches the antialias weight tables, TMA descriptors and the normalised
 * prototypes.  Not thread-safe; use one per host thread/stream set. */
int nttt_ctx_create(nttt_ctx** out, int device);
void nttt_ctx_destroy(nttt_ctx* ctx);

/* Tunables (results never depend on them).  Any other `what`, or a value out of range, returns NTTT_EINVAL.
 *   NTTT_TUNE_UPSAMPLE_STAGE_BYTES  0..160 KB: shared-memory budget per CTA of the full-resolution resize for staging the
 *                                   logit tile under its row groups (0 = every tap is read from global memory; tiles
 *                                   that do not fit take that path anyway).  Default 36 KB, the measured best on B200.
 *   NTTT_TUNE_AXIS_CACHE_ENTRIES    8..1024: capacity of the context's antialias-table cache (shrinking below the number
 *                                   held drops the cache behind a device synchronisation).  Default 1024: an image takes
 *                                   one table per distinct height and width.
 * The next two each choose between the two paths the library runs anyway, so that tests can force either one and
 * compare them bit for bit:
 *   NTTT_TUNE_LOWRES_PERSISTENT     0 or 1, process-wide.  1 (default): the low-res pass runs persistent CTAs, two per SM;
 *                                   0: one CTA per mask, the kernel the low-latency mode always runs.
 *   NTTT_TUNE_POOL_ORDER            0 or 1.  1 (default): with many images in flight (low_latency = 0) and more than 128
 *                                   masks, the pooling GEMM of nttt_match_image runs on spatially ordered rows and skips
 *                                   the k-blocks a tile of masks does not touch; 0: unordered rows without skipping, the
 *                                   path of the low-latency mode and of 128 masks or fewer. */
enum { NTTT_TUNE_UPSAMPLE_STAGE_BYTES = 1, NTTT_TUNE_AXIS_CACHE_ENTRIES = 4, NTTT_TUNE_LOWRES_PERSISTENT = 5,
       NTTT_TUNE_POOL_ORDER = 9 };
int nttt_ctx_tune(nttt_ctx* ctx, int what, long long value);

/* number of kernels this library has launched in this process (bench.py's `gpu_launches`) */
unsigned long long nttt_launch_count(void);

/* Optional per-stage CUDA-event profile of nttt_match_image: when enabled, an event is recorded on the
 * launching stream between the stage's kernels; nttt_ctx_profile_read synchronises on the last one and
 * writes the elapsed milliseconds of each stage of the most recent image to HOST memory. */
int nttt_profile_num_stages(void);
const char* nttt_profile_stage_name(int i);
int nttt_ctx_profile(nttt_ctx* ctx, int enable);
int nttt_ctx_profile_read(nttt_ctx* ctx, float* ms_host, int capacity);

/* ---------------------------------------------------------------------------------------------------
 * a6 / a9 / a15 — low-res threshold, bit-pack, area, box, stability counts
 * replaces: `lr_masks > 0` (Sam2MatchingBaseline_noAMG.py:548-549), `batched_mask_to_box(lr_masks > 0)`
 * (:614, sam2/utils/amg.py:305-348) and `calculate_stability_score` (sam2/utils/amg.py:158-178).
 *   logits [n, h, w] f32 (h*w multiple of 128; SAM-2 emits 256x256)
 *   bits   [n, h*w/32] u32          area [n] i32            box [n,4] i32 (x1,y1,x2,y2 inclusive; empty->0)
 *   stab   [n,2] i32 = {count(logit > thr+off), count(logit > thr-off)}; may be NULL (counts skipped)
 *   flags  [n] i32: bit0 = every positive logit is finite and in (2^-100, 2^100) (lets the full-res
 *          resize skip uniformly-positive footprints without evaluating them)
 */
int nttt_threshold_pack(const float* logits, int n, int h, int w, float thr, float off, uint32_t* bits,
                        int32_t* area, int32_t* box, int32_t* stab, int32_t* flags, void* stream);

/* same pass, plus the stability score AS A VALUE (`calculate_stability_score`, sam2/utils/amg.py:158-178):
 *   stab_score [n] f32 = (float)stab[i,0] / (float)stab[i,1] — torch's int32 / int32 true division in float32
 *   (counts <= h*w are exact in float32); an empty denominator gives 0/0 = NaN exactly as the reference does. */
int nttt_threshold_pack_stability(const float* logits, int n, int h, int w, float thr, float off, uint32_t* bits,
                                  int32_t* area, int32_t* box, int32_t* stab, float* stab_score, int32_t* flags,
                                  void* stream);

/* ---------------------------------------------------------------------------------------------------
 * candidate selection in front of the stage (SURVEY.md §8f rank 2)
 * replaces: `best = argmax(ious[:, 1:]) + 1; low_res_multimasks[arange, best]; ious[arange, best]`
 * (Sam2MatchingBaseline_noAMG.py:295-299), the per-batch `cat` (:423-425) and, together with `gate`, the
 * `scores_all > iou_thr` compaction (:428-431) — without moving a single logit.
 *   ious  [n, m] f32 : the decoder's predicted IoUs of its m mask planes per prompt (all batches concatenated)
 *   first            : planes [first, m) compete (the reference skips plane 0: first = 1)
 *   chunks_host      : HOST array of n_chunks DEVICE pointers (<= 64): the tensors the decoder returned, batch by
 *                      batch, each [chunk_prompts, m, h, w] f32 and 16-byte aligned (the last may hold fewer prompts)
 *   mask_ptr [n]     : device array of device pointers; mask_ptr[i] = address of prompt i's best plane
 *   score [n] f32    : = ious[i, best(i)]      (first maximal value wins; NaN counts as maximal, as torch.argmax)
 * nttt_threshold_pack_ptrs is nttt_threshold_pack reading mask i from mask_ptr[i] and skipping masks with
 * !(gate[i] > gate_min) (gate may be NULL = keep all): skipped masks are published as empty and their logits
 * are never read.
 */
int nttt_select_multimask(const float* ious, int n, int m, int first, const float* const* chunks_host, int n_chunks,
                          int chunk_prompts, int h, int w, const float** mask_ptr, float* score, void* stream);
int nttt_threshold_pack_ptrs(const float* const* mask_ptr, const float* gate, float gate_min, int n, int h, int w,
                             float thr, float off, uint32_t* bits, int32_t* area, int32_t* box, int32_t* stab,
                             int32_t* flags, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a6 (feature half) + a7 — mask-average pooling and cosine similarity
 * replaces: F.interpolate(tar_feat, 256x256, antialias) (:551-558) and compute_sim_global_avg
 * (matching_baseline_utils.py:869-904).
 *
 * Factored form: masks @ upsample(feat) == (Uy^T M Ux) @ feat.  nttt_project_masks computes the
 * [n, E] projection of each packed mask onto the encoder grid with the exact antialias weights;
 * nttt_pool_normalize contracts it with feat [E, C] on the tensor cores (split-bf16 operands, fp32
 * accumulate), divides by the area (0 -> 1) and L2-normalises (eps 1e-12).
 */
int nttt_project_masks(nttt_ctx* ctx, const uint32_t* bits, const int32_t* box /* [n,4] from threshold_pack */,
                       int n, int h, int w, int eh, int ew, float* proj /* [n, eh*ew] */, void* stream);
size_t nttt_pool_workspace_bytes(int n, int e, int c);
int nttt_pool_normalize(nttt_ctx* ctx, const float* proj, const float* feat /* [e, c] */,
                        const int32_t* area, int n, int e, int c, float* obj_feats /* [n, c] */,
                        void* workspace, size_t workspace_bytes, void* stream);

/* prototypes = normalize(mean over ALL L slots of feats_ins_avg) (matching_baseline_utils.py:893-894),
 * computed once per memory bank instead of once per image.  proto [n_cls, c] f32. */
int nttt_proto_prepare(const float* feats_ins_avg, int n_cls, int shots, int c, float* proto, void* stream);

/* a7 (similarity) + a8 (top-1 label; `k == n_cls` branch of :606-609 applies when n_cls == 1)
 *   sim [n, n_cls] f32 (may be NULL), top_score [n] f32, top_label [n] i32 (lowest index on ties) */
size_t nttt_similarity_workspace_bytes(int n, int c, int n_cls);
int nttt_similarity_top1(nttt_ctx* ctx, const float* obj_feats, const float* proto, int n, int c, int n_cls,
                         float* sim, float* top_score, int32_t* top_label, void* workspace,
                         size_t workspace_bytes, void* stream);

/* negative-reference variant of the similarity (SURVEY.md §8f rank 3; compute_sim_global_avg_with_neg,
 * matching_baseline_utils.py:906-941): sim = sp * exp(-max(sn - sp, 0) / sigma) with sp = max(obj.proto_pos[c], 0),
 * sn = max_l max(obj.proto_neg[c,l], 0).  proto_pos [n_cls, c] and proto_neg [n_cls*l_neg, c] are unit rows
 * (nttt_proto_prepare with shots = 1 normalises rows). */
size_t nttt_similarity_neg_workspace_bytes(int n, int c, int n_cls, int l_neg);
int nttt_similarity_neg_top1(nttt_ctx* ctx, const float* obj_feats, const float* proto_pos, const float* proto_neg,
                             int n, int c, int n_cls, int l_neg, float sigma, float* sim, float* top_score,
                             int32_t* top_label, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a10 / a11 — class-aware box NMS + positive-score filter
 * replaces: torchvision batched_nms(boxes.float(), pred_ious, labels, nms_thr)[:out_num] (:621-629) and the
 * `scores > 0` compaction (:631-641).  Suppression arithmetic is the published torchvision kernel's
 * (fp32 inter / (areaA + areaB - inter) > thr, areas without +1); order = score desc, index asc on ties.
 *   keep [max_keep] i32, n_keep [1] i32 : NMS survivors, truncated to max_keep (= out_num)
 *   sel  [max_keep] i32, n_sel  [1] i32 : those of `keep` whose top_score > 0, same order
 */
size_t nttt_nms_workspace_bytes(int n);
int nttt_box_nms(const int32_t* box, const float* nms_scores, const int32_t* labels, const float* top_score,
                 int n, float iou_thr, int max_keep, int32_t* keep, int32_t* n_keep, int32_t* sel,
                 int32_t* n_sel, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a12 / a9 — antialiased bilinear resize of the selected logits + threshold + bit-pack (+area, +box)
 * replaces: F.interpolate(lr_masks_out, (H,W), bilinear, antialias=True) > 0 (:657-663) and
 * batched_mask_to_box (:665).  Bit-exact with aten's arithmetic (see DESIGN.md).
 *   sel/n_sel: indices into logits (device); processes k < min(*n_sel, max_sel)
 *   bits_full [max_sel, oh, words(ow)] u32 — only words inside rect[k] are written; everything outside
 *              rect[k] is zero BY CONTRACT and must not be read
 *   rect [max_sel,4] i32 = {row0,row1,word0,word1} half-open bound derived from the low-res box
 *   area_full [max_sel] i32, box_full [max_sel,4] i32
 */
int nttt_upsample_threshold_pack(nttt_ctx* ctx, const float* logits, const uint32_t* bits_lr,
                                 const int32_t* box_lr, const int32_t* flags_lr, int ih, int iw,
                                 const int32_t* sel, const int32_t* n_sel, int max_sel, int oh, int ow,
                                 uint32_t* bits_full, int32_t* rect, int32_t* area_full, int32_t* box_full,
                                 void* stream);
/* same, with candidate i's logits at mask_ptr[i] (from nttt_select_multimask) */
int nttt_upsample_threshold_pack_ptrs(nttt_ctx* ctx, const float* const* mask_ptr, const uint32_t* bits_lr,
                                      const int32_t* box_lr, const int32_t* flags_lr, int ih, int iw,
                                      const int32_t* sel, const int32_t* n_sel, int max_sel, int oh, int ow,
                                      uint32_t* bits_full, int32_t* rect, int32_t* area_full, int32_t* box_full,
                                      void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a13 — intersection-over-self decay term on packed masks (popcount), per class
 * replaces: obj_sim = clamp(F F^T, 0) (:668-669) and compute_semantic_ios (matching_baseline_utils.py:831-867).
 *   inter_out (nullable) [max_sel, max_sel] i32 receives the integer intersection counts of same-label
 *   pairs (0 elsewhere) for parity tests.
 */
size_t nttt_mask_ios_workspace_bytes(int max_sel);
int nttt_mask_ios(const uint32_t* bits_full, const int32_t* rect, const int32_t* area_full,
                  const int32_t* box_full, const int32_t* sel, const int32_t* n_sel, int max_sel, int oh, int ow,
                  const int32_t* labels, const float* obj_feats, int c, float* ios, int32_t* inter_out,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a14 — score decay, final top-k, output gather
 * replaces: scores * pow(1 - ios, 0.5), argsort(descending)[:num_out] and the output dict (:671-683).
 * NaN sorts first (torch semantics); ties keep selection order.
 *   out_masks [num_out, oh, ow] u8 (torch.bool layout), out_boxes [num_out,4] i64, out_scores [num_out] f32,
 *   out_labels [num_out] i64, n_out [1] i32, out_index [num_out] i32 (index into logits),
 *   out_slot [num_out] i32 (position in the selected list `sel`)
 */
int nttt_decay_topk(const float* top_score, const int32_t* labels, const float* ios, const int32_t* sel,
                    const int32_t* n_sel, int max_sel, int num_out, const uint32_t* bits_full,
                    const int32_t* rect, const int32_t* box_full, int oh, int ow, uint8_t* out_masks,
                    int64_t* out_boxes, float* out_scores, int64_t* out_labels, int32_t* out_index,
                    int32_t* out_slot, int32_t* n_out, void* stream);

/* unpack all selected masks (tests / debugging): masks_u8 [max_sel, oh, ow] */
int nttt_unpack_masks(const uint32_t* bits_full, const int32_t* rect, const int32_t* n_sel, int max_sel, int oh,
                      int ow, uint8_t* masks_u8, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * result encoding after the path (SURVEY.md §8f rank 1) — COCO compressed RLE of the output masks
 * replaces: `binary_masks.cpu().numpy()` (105 MB D2H per image, pl_wrapper/sam2matcher_pl.py:144-158) followed by
 * pycocotools `mask_utils.encode(np.asfortranarray(mask))` per mask (dataset/coco_ref_dataset.py:601-604).
 * Encodes straight from the packed words; the wire format is pycocotools' rleEncode + rleToString (2.0.8):
 * column-major runs starting with zeros, then x = cnts[i] - (i > 2 ? cnts[i-2] : 0) in 5-bit groups, chars 48..111.
 *   slot (nullable) [max_count] : output j encodes packed mask slot[j] (out_slot of nttt_decay_topk); NULL: j
 *   count [1] i32 (device)      : number of live outputs; rows j >= *count get n_counts = n_chars = 0
 *   counts  [max_count, cap_counts] u32, n_counts [max_count] i32 : the uncompressed counts and their number m
 *   chars   [max_count, cap_chars]  u8,  n_chars  [max_count] i32 : the `counts` string (no terminator) and length
 * Overflow: m > cap_counts -> n_counts = m (the size needed), n_chars = -1, nothing written for that mask;
 *           length > cap_chars -> n_chars = the length needed, the string is truncated to cap_chars.
 */
int nttt_rle_encode(const uint32_t* bits_full, const int32_t* rect, const int32_t* slot, const int32_t* count,
                    int max_count, int oh, int ow, int cap_counts, int cap_chars, uint32_t* counts, int32_t* n_counts,
                    uint8_t* chars, int32_t* n_chars, void* stream);
/* Packs the strings of outputs 0..n_masks-1 back to back for one small D2H read: mask j goes to
 * out[sum_{i<j} len_i ...], len_i = n_chars[i] (a length outside [0, cap_chars] — an overflowed mask — counts as 0).
 * Replaces the per-mask `rle["counts"].decode("utf-8")` host loop's input (dataset/coco_ref_dataset.py:603-604).
 * Nothing is written past out_cap. */
int nttt_rle_compact(const uint8_t* chars, const int32_t* n_chars, int n_masks, int cap_chars, uint8_t* out,
                     int64_t out_cap, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * a2 / a5 — memory-bank fill and post-process
 * replaces: the raw-feature slot writes of forward_fill_memory (:465-485) and MemoryBank.postprocess
 * (matching_baseline_utils.py:574-599).  Instead of storing raw [n_cls,L,E,C] features the bank keeps the
 * mask-weighted sums: sum[c,l,:] = sum_e mask[e] * feat[e,:], wsum[c,l] = sum_e mask[e].
 *   soft_mask [mh, mw] f32 is nearest-resized to (eh, ew) exactly like F.interpolate(mode="nearest") (:465-469)
 *   sum_slot [c], wsum_slot [1] and mask_lowres_out [eh*ew] (nullable) are ACCUMULATED (+=): they are views of the
 *   bank slot (feats_sum[c,l], mask_sum[c,l], masks[c,l]), as `+=` at :482-484
 */
int nttt_fill_pool_accumulate(const float* feat /* [eh*ew, c] */, const float* soft_mask, int mh, int mw,
                              int eh, int ew, int c, float* sum_slot /* [c] */, float* wsum_slot /* [1] */,
                              float* mask_lowres_out, void* stream);
/* Batched form for many reference shots in ONE launch (grid = shots x column strips): feat [b, eh*ew, c],
 * soft_mask [b, mh, mw] -> sums [b, c], wsums [b], masks_lowres [b, eh*ew] (nullable); plain stores (staging rows,
 * no accumulation).  A shot pools to the same bits alone or in a batch (fixed reduction order). */
int nttt_fill_pool_batch(const float* feat, const float* soft_mask, int b, int mh, int mw, int eh, int ew, int c,
                         float* sums, float* wsums, float* masks_lowres, void* stream);
/* The slot loop of forward_fill_memory (:478-485) for n staged shots at once: dst = slot[i] (class * L + position,
 * negative = skip; destinations must be unique within a call)
 *   feats_sum[dst,:] += sums[i,:]; mask_sum[dst] += wsums[i]; masks[dst,:] += masks_lowres[i,:] (both nullable).
 * In a multi-GPU fill every rank scatters its own shots into a zero delta buffer that is then summed across ranks
 * by ONE all-reduce (replaces the three per-step all_gathers of model_utils.py:74-91). */
int nttt_fill_scatter(const float* sums, const float* wsums, const float* masks_lowres, const int32_t* slot, int n, int c,
                      int e, float* feats_sum, float* mask_sum, float* masks, void* stream);
int nttt_fill_finalize(const float* sum /* [n_cls, L, c] */, const float* wsum /* [n_cls, L] */, int n_cls,
                       int shots, int c, float* feats_ins_avg, float* feats_avg, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * The whole matching stage of one image, enqueued on one stream with no host synchronisation
 * (Sam2MatchingBaseline_noAMG.py:582-683).
 */
typedef struct nttt_match_args {
  /* inputs */
  const float* logits;    /* [n, 256, 256] */
  const float* pred_ious; /* [n] */
  const float* tar_feat;  /* [eh*ew, c] */
  const float* proto;     /* [n_cls, c] from nttt_proto_prepare */
  int32_t n, lr_h, lr_w, eh, ew, c, n_cls;
  int32_t ori_h, ori_w;
  float nms_thr;
  int32_t num_out_instance; /* outputs capacity */
  int32_t max_sel;          /* = min(8 * num_out_instance, n) */
  /* outputs (capacity num_out_instance) */
  uint8_t* out_masks;
  int64_t* out_boxes;
  float* out_scores;
  int64_t* out_labels;
  int32_t* out_index;
  int32_t* counts; /* [4] i32: n_keep, n_sel, n_out, reserved */
  /* optional taps for tests (nullable) */
  float* sim;       /* [n, n_cls] */
  float* obj_feats; /* [n, c] — if NULL, kept in workspace */
  /* workspace */
  void* workspace;
  size_t workspace_bytes;
  /* negative-reference scoring (with_negative_refs, matching_baseline_utils.py:906-941); proto_neg == NULL: off.
   * With it, `proto` must be the normalised CLASS-level average (feats_avg) and proto_neg the normalised
   * negative instance averages [n_cls * l_neg, c]; workspace from nttt_match_workspace_bytes_neg. */
  const float* proto_neg;
  int32_t l_neg;
  float sigma;
  /* fused candidate filter (Sam2MatchingBaseline_noAMG.py:428-431, `inds = scores_all > iou_thr`): when
   * filter_iou != 0, masks with !(pred_ious[i] > iou_thr) are ignored exactly as if they had been removed before the
   * stage — their logits are never read — so `logits` can be the decoder's full, un-compacted output and `n` a
   * fixed capacity (static shapes: the whole call can be captured in a CUDA graph). */
  float iou_thr;
  int32_t filter_iou;
  /* persistent outputs (nullable): out_prev_rect [num_out_instance, 4] i32, zero-initialised together with an
   * all-zero out_masks by the caller and then passed unchanged to every call that writes the SAME out_masks buffer.
   * The unpack then rewrites only the bounding box of each slot's previous and new rect instead of oh*ow bytes per
   * mask; the buffer content after the call is identical to the dense unpack's. */
  int32_t* out_prev_rect;
  /* fused multimask selection (Sam2MatchingBaseline_noAMG.py:295-299; nttt_select_multimask): when n_multi > 1,
   * the decoder's raw output is consumed in place: `multi_ious` [n, n_multi] are its predicted IoUs, `pred_ious` is
   * ignored (may be NULL); per prompt the best plane among [multi_first, n_multi) is used and its IoU becomes the
   * NMS / filter score.  The logits are either ONE buffer `logits` [n, n_multi, lr_h, lr_w] (logits_chunks_host ==
   * NULL) or the decoder's per-batch tensors: logits_chunks_host = HOST array of n_chunks (<= 64) device pointers,
   * each [chunk_prompts, n_multi, lr_h, lr_w] (`logits` is then ignored).  n_multi <= 1: off. */
  const float* multi_ious;
  int32_t n_multi;
  int32_t multi_first;
  const float* const* logits_chunks_host;
  int32_t n_chunks;
  int32_t chunk_prompts;
  /* fused result encoding (nttt_rle_encode): when rle_chars != NULL the top-`num_out_instance` masks are also emitted
   * as COCO compressed RLE, and `out_masks` may then be NULL (the dense bool masks are not produced at all).
   * Shapes as in nttt_rle_encode with max_count = num_out_instance. */
  uint32_t* rle_counts;
  int32_t* rle_n_counts;
  uint8_t* rle_chars;
  int32_t* rle_n_chars;
  int32_t rle_cap_counts;
  int32_t rle_cap_chars;
  /* scheduling hint: 0 = throughput (many images in flight on several streams: every kernel takes the launch shape that
   * costs the least SM-time — thin persistent grids of one or two CTAs per SM, no split-K — so that the kernels of
   * different images overlap: 83 us/image at 16 in flight, 330 us for one image alone);
   * 1 = low latency (one image at a time with a host synchronisation behind it, as the reference's bs=1 driver does,
   * pl_wrapper/sam2matcher_pl.py:178-191: wide grids, split-K GEMMs, the mask-independent operand preparation forked
   * onto a side stream of the context, programmatic dependent launch along the kernel chain: 204 us for one image).
   * The two modes add the fp32 partial sums of the two contractions in a different order: pooled features /
   * similarities may differ in the last bit (far inside the 1e-3 bound); every integer result (masks, boxes, counts,
   * keep lists) is computed identically. */
  int32_t low_latency;
  /* more optional taps for tests (nullable), the inputs of the score decay (a13/a14); when set, the pipeline keeps these
   * values in the caller's buffer instead of its workspace (no extra kernel), so they are what the decay and ranking read:
   *   sel       [max_sel] i32: the selection in slot order (indices into logits), after NMS and the `score > 0` filter;
   *             counts[1] entries are valid
   *   ios       [max_sel] f32: the row maximum of the intersection-over-self term that the decay reads, BEFORE the
   *             empty-mask rule: a row whose full-resolution mask is empty holds 0 here, and the decay turns it into
   *             NaN (the reference's 0/0 on the diagonal), as it does the score of that row
   *   ios_inter [max_sel, max_sel] i32: the integer intersection counts of same-label pairs of selected masks (0 on the
   *             diagonal, across labels and for disjoint boxes), as nttt_mask_ios's inter_out; zeroed by the call */
  int32_t* sel;
  float* ios;
  int32_t* ios_inter;
} nttt_match_args;

size_t nttt_match_workspace_bytes(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h,
                                  int ori_w, int max_sel);
size_t nttt_match_workspace_bytes_neg(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h,
                                      int ori_w, int max_sel, int l_neg);
int nttt_match_image(nttt_ctx* ctx, const nttt_match_args* args, void* stream);
/* sizeof(nttt_match_args) as compiled, so FFI mirrors can verify their layout */
size_t nttt_sizeof_match_args(void);

/* ---------------------------------------------------------------------------------------------------
 * The whole stage for images of any output size in a range, with the size read from device memory when the kernels
 * run: one enqueue (or one CUDA-graph capture) serves every size in [min_h, ori_h] x [min_w, ori_w].
 *   args->ori_h / ori_w are the CAPACITY (largest size); out_masks keeps the capacity's strides
 *   [num_out_instance, ori_h, ori_w], and the mask of output j occupies rows < h and columns < w of plane j.  With
 *   out_prev_rect the whole buffer equals the dense masks at (h, w) embedded top-left, zeros everywhere else (also
 *   where an earlier, larger image wrote).  Every other output is what nttt_match_image gives at ori_h = h,
 *   ori_w = w, bit for bit, in both low_latency modes.
 *   A size outside the range gives an empty result (counts[1] = counts[2] = 0, persistent slots cleared) and
 *   counts[3] = 1; otherwise counts[3] = 0.  Nothing is written outside the capacity's buffers.
 *   The first call of a range builds the resize tables of all its sizes (the context's atlas, one synchronisation);
 *   later calls with that range allocate nothing and do not synchronise.
 */
typedef struct nttt_match_size_range {
  const int32_t* ori_hw_dev; /* [2] i32, device: (h, w) of this image, read when the stage runs */
  int32_t min_h, min_w;      /* smallest size accepted (>= 1, <= the capacity) */
} nttt_match_size_range;

/* as nttt_match_workspace_bytes_neg at the capacity; 0 for an invalid range */
size_t nttt_match_workspace_bytes_sized(int n, int lr_h, int lr_w, int eh, int ew, int c, int n_cls, int ori_h,
                                        int ori_w, int max_sel, int l_neg, int min_h, int min_w);
int nttt_match_image_sized(nttt_ctx* ctx, const nttt_match_args* args, const nttt_match_size_range* range,
                           void* stream);
/* the context's resize-table atlases of the sized entry: returns their number, and (nullable outputs) their device
 * bytes and the host time their builds took in total */
int nttt_ctx_atlas_stats(nttt_ctx* ctx, size_t* bytes_host, double* build_ms_host);

/* ---------------------------------------------------------------------------------------------------
 * The whole stage with its inputs bound when it runs: the addresses of the caller's input tensors are read from a small
 * struct in DEVICE memory, so one enqueue (or one CUDA-graph capture) consumes whatever tensors a producer allocated for
 * each image, in place, with no copy into static buffers.
 *   nttt_match_bind writes the struct, stream-ordered, with one kernel that carries the values as its argument (no host
 *   staging buffer that a later bind could overwrite before it is read).  It first checks the binding against the shapes
 *   the stage was enqueued with (`shapes`: n, n_multi, n_chunks, chunk_prompts), and returns NTTT_EINVAL before any CUDA
 *   call for a null pointer, a logits base that is not 16-byte aligned (TMA bulk copies read the logits), or chunks that
 *   do not match: 1 <= n_chunks <= 64, chunk_prompts >= 1 and n_chunks * chunk_prompts >= n.
 *   nttt_match_image_bound is nttt_match_image (range == NULL) or nttt_match_image_sized with the input pointers of
 *   `args` (logits, pred_ious, multi_ious, tar_feat, logits_chunks_host) replaced by reads from `inputs_dev`; workspace,
 *   outputs and prototypes still come from `args`.  With n_multi > 1 the logits are the per-batch chunks when
 *   args->n_chunks > 0 (args->chunk_prompts prompts each), else the one buffer `logits`.  Results are those of the
 *   unbound entries on the same tensors, bit for bit.  A sized range may point `ori_hw_dev` at inputs_dev->ori_hw: the
 *   bind then writes the image's size as well.
 */
#define NTTT_MAX_CHUNKS 64
typedef struct nttt_match_inputs {
  const float* logits;     /* [n, lr_h, lr_w], or [n, n_multi, lr_h, lr_w] (n_multi > 1 without chunks) */
  const float* pred_ious;  /* [n] (n_multi <= 1) */
  const float* multi_ious; /* [n, n_multi] (n_multi > 1) */
  const float* tar_feat;   /* [eh*ew, c] */
  const float* chunks[NTTT_MAX_CHUNKS]; /* n_multi > 1 and n_chunks > 0: [chunk_prompts, n_multi, lr_h, lr_w] each */
  int32_t ori_hw[2];       /* (h, w) for a sized range that reads it */
} nttt_match_inputs;

size_t nttt_sizeof_match_inputs(void);
int nttt_match_bind(nttt_match_inputs* inputs_dev, const nttt_match_inputs* host, const nttt_match_args* shapes,
                    void* stream);
int nttt_match_image_bound(nttt_ctx* ctx, const nttt_match_args* args, const nttt_match_size_range* range,
                           const nttt_match_inputs* inputs_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NTTT_B200_H */
