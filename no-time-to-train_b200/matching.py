"""Host driver of the matching stage: one `nttt_match_image` call per image, no host synchronisation until
the caller asks for the result.

Mirrors the part of `Sam2MatchingBaselineNoAMG.forward_test` between the `_forward_sam` seam and the output
dict (`no_time_to_train/models/Sam2MatchingBaseline_noAMG.py:582-683`).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import torch

from . import _lib, ops


@dataclass
class StageConfig:
    """The `sam2_infer_cfgs` constants the stage reads (`Sam2MatchingBaseline_noAMG.py:185-194`)."""
    nms_thr: float = 0.5
    num_out_instance: int = 100
    cls_num_per_mask: int = 1
    enc_hw: tuple = (37, 37)
    expand_ratio: int = 8  # literal at :621
    neg_sigma: float = 0.8  # literal at :596 (compute_sim_global_avg_with_neg(..., sigma=0.8))
    rle_cap_counts: int = 16384  # per-mask capacity of the fused COCO-RLE output (runs / string bytes)
    rle_cap_chars: int = 32768


def _check_candidates(n: int) -> None:
    """The stage matches at most `_lib.MAX_CANDIDATES` masks per image (a 128 x 128 prompt grid); refused here, before
    anything is allocated or enqueued."""
    if n > _lib.MAX_CANDIDATES:
        raise ValueError(f"{n} candidate masks exceed the stage's limit of {_lib.MAX_CANDIDATES} per image "
                         "(points_per_side up to 128)")


@dataclass(frozen=True)
class PreparedBank:
    """One memory bank prepared for scoring (`MatchingStage.prepare_bank*`), once per bank: unit-row prototypes on the
    stage's device.  `proto` [n_cls, c] (the class-level averages when `proto_neg` is set), `proto_neg`
    [n_cls * l_neg, c] or None (plain cosine scoring)."""
    proto: torch.Tensor
    proto_neg: torch.Tensor | None
    n_cls: int
    l_neg: int
    c: int


def _check_bank(bank, capacity, c: int, device: torch.device) -> None:
    """A bank against a banked stage's capacity (n_cls, l_neg) and feature width, on the host, before anything is
    enqueued: the kernels read the prototypes' addresses and live counts from the device and check nothing."""
    if not isinstance(bank, PreparedBank):
        raise TypeError("bank must be a PreparedBank (MatchingStage.prepare_bank / prepare_bank_with_negatives)")
    cap_cls, cap_neg = capacity
    if bank.c != c:
        raise ValueError(f"the bank's prototypes have {bank.c} channels, the stage's features {c}")
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    for name, t, rows in (("proto", bank.proto, bank.n_cls), ("proto_neg", bank.proto_neg, bank.n_cls * bank.l_neg)):
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or t.device.type != "cuda" or t.device.index != dev_index:
            raise ValueError(f"bank.{name} must be a tensor on {device}")
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"bank.{name} must be contiguous float32, got {t.dtype}")
        if tuple(t.shape) != (rows, c):
            raise ValueError(f"bank.{name} has shape {tuple(t.shape)}, expected {(rows, c)}")
    if not 1 <= bank.n_cls <= cap_cls:
        raise ValueError(f"the bank has {bank.n_cls} classes, the capacity is {cap_cls}")
    if (bank.proto_neg is not None) != (cap_neg > 0):
        raise ValueError("a negative-reference bank needs a negative capacity (bank_capacity=(n_cls, l_neg > 0)), and a "
                         "plain bank a capacity without negatives")
    if cap_neg > 0 and not 1 <= bank.l_neg <= cap_neg:
        raise ValueError(f"the bank has {bank.l_neg} negatives per class, the capacity is {cap_neg}")


def _bank_capacity(bank_capacity) -> tuple:
    cap = (int(bank_capacity[0]), int(bank_capacity[1]))
    if cap[0] < 1 or cap[1] < 0:
        raise ValueError(f"bank_capacity {cap} needs n_cls >= 1 and l_neg >= 0")
    return cap


class PendingResult:
    """Device-side result of one image; `.get()` does the single D2H read of the counts and slices."""

    def __init__(self, stage, masks, boxes, scores, labels, index, counts, taps, ori_hw, keepalive, rle=None, meta=None,
                 sized=False, sim_cols=None, counted=False, rows=None):
        self._stage = stage
        self.masks, self.boxes, self.scores, self.labels, self.index = masks, boxes, scores, labels, index
        self.counts = counts
        self._meta_dev = meta if meta is not None else counts
        self._meta = None  # host copy of counts (+ the RLE lengths, which share the counts' allocation): ONE D2H read
        self.taps = taps
        self.ori_hw = ori_hw
        self._keepalive = keepalive
        self.rle = rle  # None or (counts [K,cap] i32, n_counts [K], chars [K,cap] u8, n_chars [K])
        # sized entry (`MatchingStage.graphed(..., min_hw=...)`): `masks` has the capacity's shape and `ori_hw` is the
        # size of the image the buffers hold now; the stage reports a size outside its range in counts[3]
        self._sized = sized
        self._bound = None  # a bound graph's replay: the tensors it reads (GraphedMatch.replay)
        self._bank = None  # a banked graph's replay: the bank it reads
        self._sim_cols = sim_cols  # banked: the live columns of the [n, capacity] `sim` tap
        # counted entry (`match_async(..., count_capacity=...)`, `graphed(..., counted=True)`): the taps keep the capacity's
        # rows, of which the first `rows` are this image's; the stage reports a count outside its capacity in counts[3]
        self._counted = counted
        self.rows = rows

    def rle_segmentations(self) -> list:
        """The outputs as COCO `segmentation` dicts ({"size": [h, w], "counts": str}) — what
        `mask_utils.encode(np.asfortranarray(mask))` + `.decode("utf-8")` gives in `encode_results`
        (`dataset/coco_ref_dataset.py:601-604`).  One small D2H read instead of the dense masks."""
        if self.rle is None:
            raise RuntimeError("the stage was not asked for RLE output (match_async(..., rle=True))")
        meta = self._host_meta()
        n_out = int(meta[2])
        _, n_counts, chars, n_chars = self.rle
        k = n_chars.shape[0]
        need, lens = meta[4:4 + n_out], meta[4 + k:4 + k + n_out]
        cap = chars.shape[1]
        for j, ln in enumerate(lens):
            if ln < 0 or ln > cap:
                raise RuntimeError(f"RLE of output {j} does not fit (runs needed {need[j]}, bytes needed {ln}): raise "
                                   "StageConfig.rle_cap_counts / rle_cap_chars")
        total = sum(lens)
        oh, ow = self.ori_hw
        if not total:
            return [dict(size=[oh, ow], counts="") for _ in range(n_out)]
        # the strings, packed back to back on the device and read with ONE copy of sum(len) bytes into the stage's
        # pinned staging buffer (a pageable `.cpu()` of the strided [n_out, max(len)] view costs ~0.5 ms)
        st = self._stage
        packed = st._workspace("rle_compact", chars.numel())
        _lib.check(st.lib.nttt_rle_compact(chars.data_ptr(), n_chars.data_ptr(), n_out, cap, packed.data_ptr(),
                                           packed.numel(), torch.cuda.current_stream(chars.device).cuda_stream),
                   "nttt_rle_compact")
        host = st._pinned_bytes(total)[:total]
        host.copy_(packed[:total], non_blocking=True)
        torch.cuda.current_stream(chars.device).synchronize()
        raw = host.numpy().tobytes().decode("ascii")
        out, off = [], 0
        for ln in lens:
            out.append(dict(size=[oh, ow], counts=raw[off:off + ln]))
            off += ln
        return out

    def _host_meta(self) -> list:
        if self._meta is None:
            self._meta = self._meta_dev.cpu().tolist()  # synchronises with the producing stream
        if self._sized and self._meta[3] & 1:
            raise RuntimeError(f"the stage reported status {self._meta[3]}: the image size on the device lies outside "
                               "the range the stage was enqueued for (the result is empty)")
        if self._counted and self._meta[3] & 2:
            raise RuntimeError(f"the stage reported status {self._meta[3]}: the candidate count on the device lies outside "
                               "the capacity the stage was enqueued for (the result is empty)")
        return self._meta

    def get(self) -> dict:
        counts = self._host_meta()
        n_keep, n_sel, n_out = int(counts[0]), int(counts[1]), int(counts[2])
        dev = self.boxes.device
        oh, ow = self.ori_hw
        if n_sel == 0:
            # the reference's empty early-return uses float32 zero boxes (:647-655)
            out = dict(binary_masks=torch.zeros((0, oh, ow), device=dev, dtype=torch.bool) if self.masks is not None else None,
                       bboxes=torch.zeros((0, 4), device=dev, dtype=torch.float32),
                       scores=torch.zeros((0,), device=dev, dtype=torch.float32),
                       labels=torch.zeros((0,), device=dev, dtype=torch.long))
        else:
            out = dict(binary_masks=self.masks[:n_out, :oh, :ow] if self.masks is not None else None, bboxes=self.boxes[:n_out],
                       scores=self.scores[:n_out], labels=self.labels[:n_out])
        out["counts"] = dict(n_keep=n_keep, n_sel=n_sel, n_out=n_out)
        out["index"] = self.index[:n_out]
        if self.taps:
            taps = dict(self.taps)
            if self._sim_cols is not None:
                taps["sim"] = taps["sim"][:, :self._sim_cols]
            if self._counted:
                taps["sim"], taps["obj_feats"] = taps["sim"][:self.rows], taps["obj_feats"][:self.rows]
            out["taps"] = taps
        return out


class MatchingStage:
    """Per-device matching stage.  Holds the normalised prototypes and the reusable workspace."""

    def __init__(self, device, cfg: StageConfig):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("MatchingStage needs a CUDA device: the matching stage has no CPU path")
        if cfg.cls_num_per_mask not in (1,):
            # The reference's k>1 branch passes N scores with N*k boxes to batched_nms
            # (Sam2MatchingBaseline_noAMG.py:614-629) and only works for k == 1 (k == -1 with one class).
            raise NotImplementedError("cls_num_per_mask must be 1 (or -1 with a single class)")
        self.cfg = cfg
        self.lib = _lib.load()
        self.ctx = ops.context(self.device)
        self.proto = None
        self.proto_neg = None
        self.l_neg = 0
        self.n_cls = 0
        self._ws = {}

    def prepare_bank(self, feats_ins_avg: torch.Tensor) -> PreparedBank:
        """normalize(mean over all L slots) once per bank (`matching_baseline_utils.py:893-894`)."""
        f = feats_ins_avg.to(device=self.device, dtype=torch.float32).contiguous()
        return PreparedBank(ops.proto_prepare(f), None, f.shape[0], 0, f.shape[2])

    def prepare_bank_with_negatives(self, feats_avg: torch.Tensor, feats_ins_avg_neg: torch.Tensor) -> PreparedBank:
        """Negative-reference scoring (`compute_sim_global_avg_with_neg`, `matching_baseline_utils.py:906-941`):
        positive prototypes = normalize(class-level feats_avg), negatives = normalize(every negative slot)."""
        pos = feats_avg.to(device=self.device, dtype=torch.float32).contiguous()
        neg = feats_ins_avg_neg.to(device=self.device, dtype=torch.float32).contiguous()
        n_cls, l_neg, c = neg.shape
        assert pos.shape == (n_cls, c)
        return PreparedBank(ops.proto_prepare(pos.reshape(n_cls, 1, c)), ops.proto_prepare(neg.reshape(n_cls * l_neg, 1, c)),
                            n_cls, l_neg, c)

    def set_prototypes(self, feats_ins_avg: torch.Tensor) -> None:
        """Score every later call against this bank (`prepare_bank`)."""
        self._use_bank(self.prepare_bank(feats_ins_avg))

    def set_prototypes_with_negatives(self, feats_avg: torch.Tensor, feats_ins_avg_neg: torch.Tensor) -> None:
        """Score every later call against this negative-reference bank (`prepare_bank_with_negatives`)."""
        self._use_bank(self.prepare_bank_with_negatives(feats_avg, feats_ins_avg_neg))

    def _use_bank(self, bank: PreparedBank) -> None:
        self.proto, self.proto_neg, self.l_neg, self.n_cls = bank.proto, bank.proto_neg, bank.l_neg, bank.n_cls

    def _current_bank(self) -> PreparedBank:
        if self.proto is None:
            raise RuntimeError("Memory is not ready!")  # same text as Sam2MatchingBaseline_noAMG.py:752
        return PreparedBank(self.proto, self.proto_neg, self.n_cls, self.l_neg, self.proto.shape[1])

    def _bind_bank(self, bank_dev: torch.Tensor, bank: PreparedBank, capacity) -> None:
        """Write a banked stage's device struct on the current stream (nttt_match_bank_bind: one kernel, the values in
        its argument)."""
        host = _lib.MatchBank(bank.proto.data_ptr(), ops._ptr(bank.proto_neg), bank.n_cls, bank.l_neg)
        cap = _lib.MatchArgs()
        cap.n_cls, cap.l_neg = capacity
        _lib.check(self.lib.nttt_match_bank_bind(bank_dev.data_ptr(), ctypes.byref(host), ctypes.byref(cap),
                                                 torch.cuda.current_stream(self.device).cuda_stream), "nttt_match_bank_bind")

    def _workspace(self, key, nbytes: int) -> torch.Tensor:
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty((nbytes,), dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    def match_async(self, lr_masks: torch.Tensor, pred_ious: torch.Tensor, tar_feat: torch.Tensor, ori_hw,
                    taps: bool = False, slot=0, iou_thr=None, persistent_out=None, multi_ious=None,
                    multi_first: int = 1, rle: bool = False, dense_masks: bool = True,
                    low_latency: bool = False, size_range=None, bound_inputs=None, bank=None, bank_capacity=None,
                    bank_dev=None, count_capacity=None, count_dev=None) -> PendingResult:
        """Enqueue the whole stage for one image on the current stream.  `slot` selects which reusable
        workspace to use (callers that keep several images in flight on different streams use one slot per
        stream).  `iou_thr`, if given, fuses the reference's candidate filter (`scores_all > iou_thr`,
        `Sam2MatchingBaseline_noAMG.py:428-431`): pass the decoder's full un-compacted masks and scores.
        `multi_ious` [n, m], if given, fuses the best-of-m plane selection (`:295-299`) as well: `lr_masks` is then
        the decoder's raw output — one [n, m, 256, 256] tensor, or the LIST of per-batch tensors the decoder returned
        (each [testing_point_bs, m, 256, 256]; consumed in place, no `cat`) — and `pred_ious` is ignored (pass None).
        `rle=True` also emits the outputs as COCO compressed RLE (`PendingResult.rle_segmentations()`);
        with `dense_masks=False` the bool masks are not produced at all (`binary_masks` is None).
        `taps=True` also returns the intermediate values tests compare, in `out["taps"]`: `sim`, `obj_feats` and the
        inputs of the score decay `sel`, `ios`, `ios_inter` (nttt_match_args; the counts are [max_sel, max_sel] i32).
        `low_latency=True` shapes the kernels for the shortest duration of ONE image (a caller that synchronises after
        every image) instead of the least SM-time (many images in flight); float sums may differ in the last bit between the modes.
        `size_range=(hw_dev, (min_h, min_w))` enqueues the sized entry (`nttt_match_image_sized`): `ori_hw` is then the
        capacity, and the kernels read the image's size from the device tensor `hw_dev` (int32 [2]) when they run; the
        returned result's `ori_hw` is the capacity until the caller sets it to that size (as `GraphedMatch.replay` does).
        `bound_inputs` (a device buffer of `nttt_sizeof_match_inputs()` bytes written by `nttt_match_bind`) enqueues the
        bound entry (`nttt_match_image_bound`): the kernels read the input addresses from it when they run, and the tensors
        given here only fix the shapes (as `GraphedMatch` does with `bind=True`).
        `bank_capacity=(n_cls, l_neg)` enqueues the banked entry (`nttt_match_image_banked`): the kernels read the
        prototypes and the live class count from a device struct, so the call serves any bank of up to n_cls classes
        (l_neg > 0: negative-reference banks of up to l_neg negatives per class).  `bank` (a `PreparedBank`; default: the
        stage's current prototypes) is bound into a fresh struct on the current stream; `bank_dev` (a device buffer of
        `nttt_sizeof_match_bank()` bytes) is read as it stands instead, unbound here (as `GraphedMatch` does).  The `sim`
        tap then keeps the capacity's columns on the device; `get()` returns the live ones.
        `count_capacity=N` enqueues the counted entry (`nttt_match_image_counted`): the workspace, the grids and the
        selection are sized for N candidates, and the kernels read the live count from a device int32 when they run, so
        the call serves a compacted candidate list of any length k <= N (single-plane inputs only).  The count is the
        tensors' rows, written into a fresh device int32 on the current stream; `count_dev` (a device int32 [1]) is read as
        it stands instead, unwritten here (as `GraphedMatch` does with `counted=True`).  The `sim` and `obj_feats` taps
        then keep N rows on the device; `get()` returns the first k."""
        banked = bank_capacity is not None
        if not banked and (bank is not None or bank_dev is not None):
            raise ValueError("bank= and bank_dev= need bank_capacity=(n_cls, l_neg)")
        if banked:
            cap = _bank_capacity(bank_capacity)
            if bank_dev is None:
                bank = bank if bank is not None else self._current_bank()
                _check_bank(bank, cap, tar_feat.shape[-1], self.device)
        elif self.proto is None:
            raise RuntimeError("Memory is not ready!")  # same text as Sam2MatchingBaseline_noAMG.py:752
        n_cls, l_neg = cap if banked else (self.n_cls, self.l_neg)
        ops._need(tar_feat, torch.float32, "tar_feat")
        n_multi, chunks = 0, None
        if multi_ious is not None:
            ops._need(multi_ious, torch.float32, "multi_ious")
            chunks = list(lr_masks) if isinstance(lr_masks, (list, tuple)) else [lr_masks]
            n, n_multi = multi_ious.shape
            bs, _, lh, lw = chunks[0].shape
            for i, ch in enumerate(chunks):
                ops._need(ch, torch.float32, "lr_masks chunk")
                if ch.dim() != 4 or tuple(ch.shape[1:]) != (n_multi, lh, lw) or (ch.shape[0] != bs and i + 1 < len(chunks)):
                    raise ValueError("with multi_ious [n, m], lr_masks must be the decoder's [bs, m, h, w] outputs")
            if sum(ch.shape[0] for ch in chunks) != n:
                raise ValueError("multi_ious rows must match the prompts in lr_masks")
            if n_multi < 2 or not 0 <= multi_first < n_multi:
                raise ValueError("multi_ious needs m >= 2 planes and 0 <= multi_first < m")
        else:
            ops._need(lr_masks, torch.float32, "lr_masks")
            ops._need(pred_ious, torch.float32, "pred_ious")
            n, lh, lw = lr_masks.shape
        _check_candidates(n)
        counted = count_capacity is not None
        rows = n  # the candidates this call's tensors hold (counted: the live count k)
        if counted:
            if n_multi:
                raise ValueError("the counted entry takes single-plane candidates (compacted lists), not multi_ious")
            n = int(count_capacity)
            _check_candidates(n)
            if not 0 <= rows <= n:
                raise ValueError(f"{rows} candidates exceed the count capacity {n}")
        elif count_dev is not None:
            raise ValueError("count_dev= needs count_capacity=N")
        eh, ew = self.cfg.enc_hw
        e, c = tar_feat.shape
        if e != eh * ew:
            raise ValueError(f"tar_feat has {e} patches, expected {eh}x{ew}")
        oh, ow = int(ori_hw[0]), int(ori_hw[1])
        if size_range is not None:
            hw_dev, (min_h, min_w) = size_range[0], (int(size_range[1][0]), int(size_range[1][1]))
            if hw_dev.dtype != torch.int32 or hw_dev.numel() != 2 or hw_dev.device != self.device:
                raise ValueError("size_range needs an int32 [2] tensor on the stage's device")
            if not (1 <= min_h <= oh and 1 <= min_w <= ow):
                raise ValueError(f"min_hw {(min_h, min_w)} must lie between 1 and the capacity {(oh, ow)}")
        num_out = int(self.cfg.num_out_instance)
        max_sel = int(min(num_out * self.cfg.expand_ratio, n))
        dev = self.device
        prev_rect = None
        if not dense_masks:
            if not rle:
                raise ValueError("dense_masks=False needs rle=True")
            masks = None
        elif persistent_out is not None:
            # outputs owned by the caller and reused call after call: (masks u8 [num_out,oh,ow] zero-initialised,
            # prev_rect i32 [num_out,4] zero-initialised); only the changed rectangles are rewritten
            masks, prev_rect = persistent_out
            assert masks.shape == (max(num_out, 1), oh, ow) and masks.dtype == torch.uint8
        else:
            masks = torch.empty((max(num_out, 1), oh, ow), dtype=torch.uint8, device=dev)
        # (no fills: only the first n_out rows are ever read, and the pipeline writes the counts itself)
        boxes = torch.empty((max(num_out, 1), 4), dtype=torch.int64, device=dev)
        scores = torch.empty((max(num_out, 1),), dtype=torch.float32, device=dev)
        labels = torch.empty((max(num_out, 1),), dtype=torch.int64, device=dev)
        index = torch.empty((max(num_out, 1),), dtype=torch.int32, device=dev)
        k_rle = max(num_out, 1) if rle else 0
        meta = torch.empty((4 + 2 * k_rle,), dtype=torch.int32, device=dev)  # counts | rle n_counts | rle n_chars
        counts = meta[:4]
        tap_t = {}
        if taps:
            tap_t["sim"] = torch.empty((n, n_cls), dtype=torch.float32, device=dev)
            tap_t["obj_feats"] = torch.empty((n, c), dtype=torch.float32, device=dev)
            # the inputs of the score decay: selection in slot order, IoS row maxima, same-label intersection counts
            tap_t["sel"] = torch.empty((max(max_sel, 1),), dtype=torch.int32, device=dev)
            tap_t["ios"] = torch.empty((max(max_sel, 1),), dtype=torch.float32, device=dev)
            tap_t["ios_inter"] = torch.empty((max(max_sel, 1), max(max_sel, 1)), dtype=torch.int32, device=dev)
        if size_range is None:
            ws_bytes = self.lib.nttt_match_workspace_bytes_neg(n, lh, lw, eh, ew, c, n_cls, oh, ow, max_sel, l_neg)
        else:
            ws_bytes = self.lib.nttt_match_workspace_bytes_sized(n, lh, lw, eh, ew, c, n_cls, oh, ow, max_sel, l_neg,
                                                                 min_h, min_w)
        ws = self._workspace(("match", slot), ws_bytes)
        a = _lib.MatchArgs()
        a.logits, a.pred_ious, a.tar_feat = None if chunks else lr_masks.data_ptr(), ops._ptr(pred_ious), tar_feat.data_ptr()
        empty_rows = None
        if counted and rows == 0:
            # an empty compacted list (`masks[keep]` with nothing kept) may have no address at all; the stage reads no
            # row of it, so any valid 16-byte-aligned buffer stands in
            empty_rows = torch.empty((4,), dtype=torch.float32, device=dev)
            a.logits = a.pred_ious = empty_rows.data_ptr()
        a.proto = None if banked else self.proto.data_ptr()
        a.multi_ious, a.n_multi, a.multi_first = ops._ptr(multi_ious), n_multi, int(multi_first)
        if chunks:
            table = ops.chunk_table(chunks)
            a.logits_chunks_host, a.n_chunks, a.chunk_prompts = table, len(chunks), int(chunks[0].shape[0])
        a.n, a.lr_h, a.lr_w, a.eh, a.ew, a.c, a.n_cls = n, lh, lw, eh, ew, c, n_cls
        a.ori_h, a.ori_w = oh, ow
        a.nms_thr = float(self.cfg.nms_thr)
        a.num_out_instance, a.max_sel = num_out, max_sel
        a.out_masks, a.out_boxes, a.out_scores, a.out_labels = (ops._ptr(masks), boxes.data_ptr(),
                                                                scores.data_ptr(), labels.data_ptr())
        rle_t = None
        if rle:
            k, cc, ch = max(num_out, 1), int(self.cfg.rle_cap_counts), int(self.cfg.rle_cap_chars)
            rle_t = (torch.empty((k, cc), dtype=torch.int32, device=dev), meta[4:4 + k],
                     torch.empty((k, ch), dtype=torch.uint8, device=dev), meta[4 + k:])
            a.rle_counts, a.rle_n_counts, a.rle_chars, a.rle_n_chars = (t.data_ptr() for t in rle_t)
            a.rle_cap_counts, a.rle_cap_chars = cc, ch
        a.out_index, a.counts = index.data_ptr(), counts.data_ptr()
        a.sim = tap_t["sim"].data_ptr() if taps else None
        a.obj_feats = tap_t["obj_feats"].data_ptr() if taps else None
        a.sel, a.ios, a.ios_inter = ((tap_t[k].data_ptr() for k in ("sel", "ios", "ios_inter")) if taps
                                     else (None, None, None))
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.proto_neg = self.proto_neg.data_ptr() if self.proto_neg is not None and not banked else None
        a.l_neg, a.sigma = l_neg, float(self.cfg.neg_sigma)
        a.iou_thr, a.filter_iou = (float(iou_thr), 1) if iou_thr is not None else (0.0, 0)
        a.out_prev_rect = prev_rect.data_ptr() if prev_rect is not None else None
        a.low_latency = 1 if low_latency else 0
        stream = torch.cuda.current_stream(dev).cuda_stream
        rng = _lib.MatchSizeRange(hw_dev.data_ptr(), min_h, min_w) if size_range is not None else None
        if banked and bank_dev is None:
            bank_dev = torch.empty((int(self.lib.nttt_sizeof_match_bank()),), dtype=torch.uint8, device=dev)
            self._bind_bank(bank_dev, bank, cap)
        if counted:
            if count_dev is None:
                count_dev = torch.empty((1,), dtype=torch.int32, device=dev)
                self._bind_count(count_dev, rows, n)
            elif count_dev.dtype != torch.int32 or count_dev.numel() != 1 or count_dev.device != dev:
                raise ValueError("count_dev must be an int32 [1] tensor on the stage's device")
            _lib.check(self.lib.nttt_match_image_counted(self.ctx, ctypes.byref(a), ctypes.byref(rng) if rng else None,
                                                         ops._ptr(bound_inputs), ops._ptr(bank_dev), count_dev.data_ptr(),
                                                         stream), "nttt_match_image_counted")
        elif banked:
            _lib.check(self.lib.nttt_match_image_banked(self.ctx, ctypes.byref(a), ctypes.byref(rng) if rng else None,
                                                        ops._ptr(bound_inputs), bank_dev.data_ptr(), stream),
                       "nttt_match_image_banked")
        elif bound_inputs is not None:
            _lib.check(self.lib.nttt_match_image_bound(self.ctx, ctypes.byref(a), ctypes.byref(rng) if rng else None,
                                                       bound_inputs.data_ptr(), stream), "nttt_match_image_bound")
        elif size_range is None:
            _lib.check(self.lib.nttt_match_image(self.ctx, ctypes.byref(a), stream), "nttt_match_image")
        else:
            _lib.check(self.lib.nttt_match_image_sized(self.ctx, ctypes.byref(a), ctypes.byref(rng), stream),
                       "nttt_match_image_sized")
        return PendingResult(self, masks.view(torch.bool) if masks is not None else None, boxes, scores, labels, index,
                             counts, tap_t, (oh, ow), keepalive=(lr_masks, pred_ious, multi_ious, tar_feat, ws, size_range, empty_rows,
                                                                bound_inputs, bank, bank_dev, count_dev),
                             rle=rle_t, meta=meta, sized=size_range is not None,
                             sim_cols=bank.n_cls if banked and bank is not None else None, counted=counted, rows=rows)

    def _bind_count(self, count_dev: torch.Tensor, k: int, capacity: int) -> None:
        """Write a counted stage's live count on the current stream (nttt_match_count_bind: one kernel, the value in its
        argument)."""
        cap = _lib.MatchArgs()
        cap.n = int(capacity)
        _lib.check(self.lib.nttt_match_count_bind(count_dev.data_ptr(), int(k), ctypes.byref(cap),
                                                  torch.cuda.current_stream(self.device).cuda_stream),
                   "nttt_match_count_bind")

    def atlas_stats(self) -> dict:
        """The resize-table atlases the sized graphs of this device's context use: count, device bytes, build time."""
        nbytes, ms = ctypes.c_size_t(0), ctypes.c_double(0.0)
        n = self.lib.nttt_ctx_atlas_stats(self.ctx, ctypes.byref(nbytes), ctypes.byref(ms))
        if n < 0:
            _lib.check(n, "nttt_ctx_atlas_stats")
        return dict(atlases=n, bytes=int(nbytes.value), build_ms=float(ms.value))

    def _pinned_bytes(self, nbytes: int) -> torch.Tensor:
        """Pinned host staging for result reads (grown on demand, reused call after call)."""
        buf = self._ws.get("pinned")
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty((max(nbytes, 1 << 20),), dtype=torch.uint8).pin_memory()
            self._ws["pinned"] = buf
        return buf

    TUNABLES = {"upsample_stage_bytes": 1, "axis_cache_entries": 4, "lowres_persistent": 5,
                "pool_order": 9}  # include/nttt_b200.h: NTTT_TUNE_*

    def tune(self, name: str, value: int) -> None:
        """Set a tunable of this device's context (`nttt_ctx_tune`); results never depend on them."""
        if name not in self.TUNABLES:
            raise ValueError(f"unknown tunable {name!r}; known: {', '.join(self.TUNABLES)}")
        _lib.check(self.lib.nttt_ctx_tune(self.ctx, self.TUNABLES[name], int(value)), f"nttt_ctx_tune({name})")

    def profile(self, enable: bool) -> None:
        """Per-stage CUDA-event timing of the next `match_async` calls (see nttt_ctx_profile)."""
        _lib.check(self.lib.nttt_ctx_profile(self.ctx, int(enable)), "nttt_ctx_profile")

    def profile_read(self) -> dict:
        """Stage name -> milliseconds of the most recent image (synchronises on its last event)."""
        n = self.lib.nttt_profile_num_stages()
        buf = (ctypes.c_float * n)()
        got = self.lib.nttt_ctx_profile_read(self.ctx, buf, n)
        if got < 0:
            _lib.check(got, "nttt_ctx_profile_read")
        return {self.lib.nttt_profile_stage_name(i).decode(): float(buf[i]) for i in range(got)}

    def match(self, lr_masks, pred_ious, tar_feat, ori_hw, taps: bool = False, iou_thr=None, multi_ious=None,
              multi_first: int = 1, rle: bool = False, dense_masks: bool = True, persistent_out=None,
              low_latency: bool = True) -> dict:
        """One image, synchronously (the caller waits for the result): runs in low-latency mode by default."""
        pend = self.match_async(lr_masks, pred_ious, tar_feat, ori_hw, taps=taps, iou_thr=iou_thr,
                                multi_ious=multi_ious, multi_first=multi_first, rle=rle, dense_masks=dense_masks,
                                persistent_out=persistent_out, low_latency=low_latency)
        out = pend.get()
        if rle:
            out["segmentations"] = pend.rle_segmentations()
        return out

    def graphed(self, n: int, c: int, ori_hw, iou_thr=None, key=None, n_multi: int = 0,
                multi_first: int = 1, rle: bool = False, dense_masks: bool = True, persistent_out=None,
                low_latency: bool = False, min_hw=None, bind: bool = False, chunk_prompts=None,
                bank_capacity=None, counted: bool = False) -> "GraphedMatch":
        """A CUDA-graph capture of the whole stage at fixed shapes with static input/output buffers.
        n_multi > 1: the static mask buffer is the decoder's raw [n, n_multi, 256, 256] output (+ `multi_ious`).
        rle / dense_masks: as in `match_async`.  `key` names the workspace slot and `persistent_out` the
        (masks, prev_rect) output buffers: graphs that are replayed on the SAME stream may share both (a caller
        holding one graph per resident image passes the stream's slot).  `low_latency`: capture the launch shapes
        for one image at a time (a caller that waits for each result) instead of many images in flight.
        `min_hw=(h, w)`: one graph for every output size between `min_hw` and `ori_hw` (the capacity); the size of each
        image is given to `replay(ori_hw=...)`, which writes it to the device, and the kernels read it when they run.
        `bind=True`: the graph reads its inputs' addresses on the device, so `replay(lr_masks=..., pred_ious=...,
        multi_ious=..., tar_feat=...)` consumes a producer's own tensors in place (see `GraphedMatch.replay`).
        `chunk_prompts` (with n_multi > 1): the static masks are the decoder's per-batch chunk list, `chunk_prompts`
        prompts each (the last holds the rest), instead of one [n, n_multi, 256, 256] tensor.
        `bank_capacity=(n_cls, l_neg)`: the graph reads its memory bank on the device, so `replay(bank=...)` scores the
        image against any `PreparedBank` of up to n_cls classes (and, with l_neg > 0, up to l_neg negatives per class)
        without a new capture (see `GraphedMatch.replay`).
        `counted=True`: `n` is a capacity; the graph reads the live candidate count on the device, so `replay(n=k)` (or,
        bound, `replay(lr_masks=[k, 256, 256], pred_ious=[k])`) serves a compacted candidate list of any length
        0 <= k <= n without a new capture (single-plane inputs only)."""
        return GraphedMatch(self, n, c, ori_hw, iou_thr, key, n_multi, multi_first, rle, dense_masks, persistent_out,
                            low_latency, min_hw, bind, chunk_prompts, bank_capacity, counted)


class GraphedMatch:
    """The stage of one image captured once into a CUDA graph and replayed with one launch.

    Shapes are static: `n` is a fixed capacity (e.g. points_per_side**2) and the fused `iou_thr` filter takes the
    place of the reference's compaction, so the producer writes the decoder's masks / scores and the encoder's
    features straight into `self.lr_masks`, `self.pred_ious`, `self.tar_feat` (static device buffers) and calls
    `replay()`.  Outputs live in static buffers too: consume a result (`.get()`) before replaying the same object
    again.  Replay costs one graph launch on the host instead of ~18 kernel launches.

    With `min_hw` the graph is SIZED: `ori_hw` is the capacity, the output masks keep its shape (image j's mask in the
    top-left [h, w] corner of plane j, zeros elsewhere) and `replay(ori_hw=(h, w))` serves any size in between.

    With `bind=True` the graph is BOUND: it reads the addresses of its inputs from a small device struct
    (`nttt_match_inputs`) that `replay(lr_masks=..., ...)` rewrites with one kernel on the replay's stream, so each replay
    consumes the producer's own tensors in place.  Until a replay binds something else, the binding points at the graph's
    own static buffers.

    With `bank_capacity` the graph is BANKED: it reads the prototypes' addresses and the live class count from a small
    device struct (`nttt_match_bank`) that every replay rewrites with one kernel on the replay's stream, so one capture
    serves every bank up to the capacity, and `set_prototypes*` never makes it re-capture.

    With `counted=True` the graph is COUNTED: `n` is a capacity, and every replay writes the live candidate count k to a
    device int32 with one kernel on the replay's stream; the kernels read it and touch no candidate at or past it.

    An unbanked graph keeps the prototype tensors it captured alive, and re-captures on the next replay once the stage's
    prototypes have been replaced (`set_prototypes*`)."""

    def __init__(self, stage: MatchingStage, n: int, c: int, ori_hw, iou_thr=None, key=None, n_multi: int = 0,
                 multi_first: int = 1, rle: bool = False, dense_masks: bool = True, persistent_out=None,
                 low_latency: bool = False, min_hw=None, bind: bool = False, chunk_prompts=None, bank_capacity=None,
                 counted: bool = False):
        dev = stage.device
        eh, ew = stage.cfg.enc_hw
        _check_candidates(int(n))
        if counted and n_multi > 1:
            raise ValueError("a counted graph takes single-plane candidates (compacted lists): n_multi must be <= 1")
        self.counted = bool(counted)
        self.count_dev = torch.zeros((1,), dtype=torch.int32, device=dev) if self.counted else None
        self.stage = stage
        self.n, self.c = int(n), int(c)
        self.n_multi = int(n_multi) if n_multi > 1 else 0
        self.chunk_prompts = None
        if n_multi > 1:
            full = torch.zeros((n, n_multi, 256, 256), dtype=torch.float32, device=dev)
            if chunk_prompts is not None:
                cp = int(chunk_prompts)
                if cp < 1 or -(-n // cp) > _lib.MAX_CHUNKS:
                    raise ValueError(f"chunk_prompts {chunk_prompts} must split {n} prompts into 1..{_lib.MAX_CHUNKS} chunks")
                self.chunk_prompts = cp
                self.lr_masks = list(full.split(cp))  # (views of one buffer: the decoder's per-batch layout)
            else:
                self.lr_masks = full
            self.multi_ious = torch.zeros((n, n_multi), dtype=torch.float32, device=dev)
            self.pred_ious = None
        else:
            if chunk_prompts is not None:
                raise ValueError("chunk_prompts needs n_multi > 1 (the decoder's raw multimask outputs)")
            self.lr_masks = torch.zeros((n, 256, 256), dtype=torch.float32, device=dev)
            self.pred_ious = torch.zeros((n,), dtype=torch.float32, device=dev)
            self.multi_ious = None
        self.multi_first = multi_first
        self._kw = dict(rle=rle, dense_masks=dense_masks, low_latency=low_latency)
        self.tar_feat = torch.zeros((eh * ew, c), dtype=torch.float32, device=dev)
        self.ori_hw = (int(ori_hw[0]), int(ori_hw[1]))
        self.bind = bool(bind)
        self.inputs_dev = None
        if self.bind:
            lib = stage.lib
            self.inputs_dev = torch.zeros((int(lib.nttt_sizeof_match_inputs()),), dtype=torch.uint8, device=dev)
            # the shapes every binding is checked against (nttt_match_bind)
            self._shapes = _lib.MatchArgs()
            self._shapes.n, self._shapes.n_multi = self.n, self.n_multi
            if self.n_multi:
                k = len(self.lr_masks) if self.chunk_prompts else 1
                self._shapes.n_chunks, self._shapes.chunk_prompts = k, self.chunk_prompts or self.n
            self._static_bound = False  # the device struct holds the static buffers' addresses
        self.min_hw = None
        self._size_range = None
        if min_hw is not None:
            self.min_hw = (int(min_hw[0]), int(min_hw[1]))
            if not (1 <= self.min_hw[0] <= self.ori_hw[0] and 1 <= self.min_hw[1] <= self.ori_hw[1]):
                raise ValueError(f"min_hw {self.min_hw} must lie between 1 and the capacity {self.ori_hw}")
            if self.bind:
                # the size the kernels read is part of the bound struct: one bind kernel writes inputs and size
                off = _lib.MatchInputs.ori_hw.offset
                self.hw_dev = self.inputs_dev[off:off + 8].view(torch.int32)
            else:
                # the size the kernels read; replay() rewrites it, stream-ordered, before each launch of the graph
                self.hw_dev = torch.tensor(self.ori_hw, dtype=torch.int32, device=dev)
            self._size_range = (self.hw_dev, self.min_hw)
        self.iou_thr = iou_thr
        self._slot = ("graph", id(self) if key is None else key)
        num_out = max(int(stage.cfg.num_out_instance), 1)
        # persistent outputs: the mask buffer is zeroed once; afterwards every replay rewrites only the rectangles
        # that change (nttt_match_args.out_prev_rect)
        if persistent_out is not None and dense_masks:
            self._out = persistent_out
        else:
            self._out = (torch.zeros((num_out, self.ori_hw[0], self.ori_hw[1]), dtype=torch.uint8, device=dev),
                         torch.zeros((num_out, 4), dtype=torch.int32, device=dev)) if dense_masks else None
        self.bank_capacity = None
        self.bank_dev = None
        if bank_capacity is not None:
            self.bank_capacity = _bank_capacity(bank_capacity)
            self.bank_dev = torch.zeros((int(stage.lib.nttt_sizeof_match_bank()),), dtype=torch.uint8, device=dev)
        self.graph = None
        self.pending = None
        self._proto = None  # unbanked: the prototype tensors the graph was captured with (its kernels read their addresses)

    def _static_inputs(self) -> dict:
        return dict(lr_masks=self.lr_masks, pred_ious=self.pred_ious, multi_ious=self.multi_ious, tar_feat=self.tar_feat)

    def _bind(self, inputs: dict, hw) -> None:
        """Write the device struct on the current stream (nttt_match_bind: one kernel, the values in its argument)."""
        host = _lib.MatchInputs()
        lr = inputs["lr_masks"]
        if self.n_multi:
            for i, t in enumerate(lr if isinstance(lr, list) else [lr]):
                host.chunks[i] = t.data_ptr()
            host.multi_ious = inputs["multi_ious"].data_ptr()
        else:
            host.logits, host.pred_ious = lr.data_ptr(), inputs["pred_ious"].data_ptr()
        host.tar_feat = inputs["tar_feat"].data_ptr()
        host.ori_hw[0], host.ori_hw[1] = int(hw[0]), int(hw[1])
        stream = torch.cuda.current_stream(self.stage.device).cuda_stream
        _lib.check(self.stage.lib.nttt_match_bind(self.inputs_dev.data_ptr(), ctypes.byref(host),
                                                  ctypes.byref(self._shapes), stream), "nttt_match_bind")

    def _check_bound(self, lr_masks, pred_ious, multi_ious, tar_feat, k=None) -> dict:
        """The tensors a replay binds (the static buffers where one is not given), checked against the capture's shapes
        on the host: dtype, device, contiguity, shape and the 16-byte alignment of every logits base.  A counted graph
        takes k candidate rows (its static buffers' first k where no tensor is given)."""
        dev = self.stage.device
        dev_index = dev.index if dev.index is not None else torch.cuda.current_device()

        def need(t, shape, name):
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"{name} must be a tensor")
            if t.device.type != "cuda" or t.device.index != dev_index:
                raise ValueError(f"{name} must be on {dev} (the graph's device), got {t.device}")
            ops._need(t, torch.float32, name)
            if tuple(t.shape) != tuple(shape):
                raise ValueError(f"{name} has shape {tuple(t.shape)}, the graph was captured for {tuple(shape)}")
            return t

        def aligned(t, name):
            if t.data_ptr() % 16:
                raise ValueError(f"{name} must start on a 16-byte boundary (the low-res pass reads it with TMA bulk "
                                 "copies)")
            return t

        got = self._static_inputs()
        if k is not None:
            got["lr_masks"], got["pred_ious"] = got["lr_masks"][:k], got["pred_ious"][:k]
        if tar_feat is not None:
            got["tar_feat"] = need(tar_feat, self.tar_feat.shape, "tar_feat")
        if self.n_multi:
            if pred_ious is not None:
                raise ValueError("a multimask graph takes multi_ious, not pred_ious")
            if multi_ious is not None:
                got["multi_ious"] = need(multi_ious, self.multi_ious.shape, "multi_ious")
            if lr_masks is not None:
                if self.chunk_prompts:
                    if not isinstance(lr_masks, (list, tuple)) or len(lr_masks) != len(self.lr_masks):
                        raise ValueError(f"lr_masks must be the decoder's list of {len(self.lr_masks)} per-batch chunks")
                    got["lr_masks"] = [aligned(need(t, ref.shape, f"lr_masks chunk {i}"), f"lr_masks chunk {i}")
                                       for i, (t, ref) in enumerate(zip(lr_masks, self.lr_masks))]
                else:
                    got["lr_masks"] = aligned(need(lr_masks, self.lr_masks.shape, "lr_masks"), "lr_masks")
        else:
            if multi_ious is not None:
                raise ValueError("a single-plane graph takes pred_ious, not multi_ious")
            if pred_ious is not None:
                got["pred_ious"] = need(pred_ious, got["pred_ious"].shape, "pred_ious")
            if lr_masks is not None:
                got["lr_masks"] = aligned(need(lr_masks, got["lr_masks"].shape, "lr_masks"), "lr_masks")
        return got

    def capture(self, bank=None):
        """Warm up (workspace allocation, antialias tables) on a side stream, then capture.  A banked graph's warm-up
        reads `bank` (default: the stage's current prototypes)."""
        st = self.stage
        if self.bind:
            self._bind(self._static_inputs(), self.ori_hw)
            self._static_bound = True
        kw = dict(slot=self._slot, iou_thr=self.iou_thr, persistent_out=self._out, multi_ious=self.multi_ious,
                  multi_first=self.multi_first, size_range=self._size_range, bound_inputs=self.inputs_dev, **self._kw)
        if self.bank_capacity is not None:
            bank = bank if bank is not None else st._current_bank()
            _check_bank(bank, self.bank_capacity, self.c, st.device)
            st._bind_bank(self.bank_dev, bank, self.bank_capacity)
            kw.update(bank_capacity=self.bank_capacity, bank_dev=self.bank_dev)
        if self.counted:
            st._bind_count(self.count_dev, self.n, self.n)  # (the warm-up and the capture read the static buffers)
            kw.update(count_capacity=self.n, count_dev=self.count_dev)
        side = torch.cuda.Stream(st.device)
        side.wait_stream(torch.cuda.current_stream(st.device))
        with torch.cuda.stream(side):
            for _ in range(2):
                st.match_async(self.lr_masks, self.pred_ious, self.tar_feat, self.ori_hw, **kw)
        torch.cuda.current_stream(st.device).wait_stream(side)
        torch.cuda.synchronize(st.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.pending = st.match_async(self.lr_masks, self.pred_ious, self.tar_feat, self.ori_hw, **kw)
        self._proto = (st.proto, st.proto_neg)
        return self

    def replay(self, ori_hw=None, lr_masks=None, pred_ious=None, multi_ious=None, tar_feat=None, bank=None,
               n=None) -> PendingResult:
        """Launch the graph on the current stream.  A sized graph needs the image's size `ori_hw=(h, w)`.

        A bound graph (`bind=True`) also takes the image's inputs: `lr_masks` (a tensor, or with `chunk_prompts` the
        decoder's list of per-batch chunks), `pred_ious` or `multi_ious`, and `tar_feat`, each float32, contiguous, on the
        graph's device and of the capture's shape; an input not given is the graph's own static buffer.  Everything is
        checked before anything is enqueued.  The replay reads the tensors on the current stream: a producer that wrote
        them on another stream must make this stream wait for it first (`torch.cuda.current_stream().wait_stream(p)`).
        The result holds them until the graph's next replay.

        A banked graph (`bank_capacity`) scores against `bank`, a `PreparedBank` of the graph's channel count, device
        and kind (negative references or not) with no more classes or negatives than the capacity, or, without one,
        against the stage's current prototypes.  It is checked before anything is enqueued, bound on the current stream
        and held by the result until the graph's next replay.

        A counted graph (`counted=True`) matches k candidates, 0 <= k <= the capacity `n` of the capture: bound, the
        given `lr_masks` [k, 256, 256] and `pred_ious` [k] (both, with the same k); otherwise `n=k` of its inputs' rows
        (the static buffers' first k), by default all of them.  k is checked before anything is enqueued and written to
        the device on the current stream; `get()` slices the `sim` / `obj_feats` taps to k rows."""
        given = lr_masks is not None or pred_ious is not None or multi_ious is not None or tar_feat is not None
        k = None
        if self.counted:
            if (lr_masks is None) != (pred_ious is None):
                raise ValueError("a counted graph takes lr_masks and pred_ious together (their rows are the count)")
            if lr_masks is not None:
                if not isinstance(lr_masks, torch.Tensor) or not isinstance(pred_ious, torch.Tensor):
                    raise TypeError("lr_masks and pred_ious must be tensors")
                k = int(lr_masks.shape[0])
                if pred_ious.dim() != 1 or int(pred_ious.shape[0]) != k:
                    raise ValueError(f"pred_ious has shape {tuple(pred_ious.shape)}, lr_masks {k} rows")
                if n is not None and int(n) != k:
                    raise ValueError(f"n={n} does not match the {k} rows of lr_masks")
            else:
                k = self.n if n is None else int(n)
            if not 0 <= k <= self.n:
                raise ValueError(f"{k} candidates are outside the graph's count capacity 0 .. {self.n}")
        elif n is not None:
            raise ValueError("this graph serves its capture's candidate count only; capture it with counted=True")
        if given and not self.bind:
            raise ValueError("this graph reads its static buffers; capture it with bind=True to pass inputs to replay()")
        banked = self.bank_capacity is not None
        if bank is not None and not banked:
            raise ValueError("this graph reads the prototypes it was captured with; capture it with bank_capacity to pass "
                             "a bank to replay()")
        if self.min_hw is None:
            if ori_hw is not None and (int(ori_hw[0]), int(ori_hw[1])) != self.ori_hw:
                raise ValueError(f"this graph serves {self.ori_hw} only; capture it with min_hw to serve a range")
            hw = self.ori_hw
        else:
            if ori_hw is None:
                raise ValueError("a sized graph needs the image's size: replay(ori_hw=(h, w))")
            hw = (int(ori_hw[0]), int(ori_hw[1]))
            if not (self.min_hw[0] <= hw[0] <= self.ori_hw[0] and self.min_hw[1] <= hw[1] <= self.ori_hw[1]):
                raise ValueError(f"size {hw} is outside the graph's range {self.min_hw} .. {self.ori_hw}")
        # (without tensors a bound graph reads its static buffers, whose first k rows start where all of them do)
        inputs = self._check_bound(lr_masks, pred_ious, multi_ious, tar_feat, k) if given else None
        if inputs is not None and k == 0:  # (an empty list has no address to bind; no row of the static ones is read)
            inputs.update(lr_masks=self.lr_masks, pred_ious=self.pred_ious)
        st = self.stage
        if banked:
            bank = bank if bank is not None else st._current_bank()
            _check_bank(bank, self.bank_capacity, self.c, st.device)
        if self.graph is None or (not banked and (self._proto[0] is not st.proto or self._proto[1] is not st.proto_neg)):
            self.capture(bank)  # (first replay, or the stage's prototypes were replaced since an unbanked capture)
        if self.bind:
            if given or self.min_hw is not None or not self._static_bound:
                self._bind(inputs or self._static_inputs(), hw)
                self._static_bound = not given
        elif self.min_hw is not None:
            # One fill kernel on the replay's stream writes both int32 (little-endian: h is the low half): the value
            # travels as a kernel argument, so no host buffer can be overwritten by a later replay before it is read.
            self.hw_dev.view(torch.int64).fill_(hw[0] | (hw[1] << 32))
        if banked:
            st._bind_bank(self.bank_dev, bank, self.bank_capacity)
        if self.counted:
            st._bind_count(self.count_dev, k, self.n)
        self.graph.replay()
        self.pending._meta = None  # the static buffers now hold a new image's result
        self.pending.ori_hw = hw
        self.pending._bound = inputs  # (the tensors this replay reads, held until the next one)
        self.pending._bank = bank
        self.pending.rows = k if self.counted else self.pending.rows
        return self.pending
