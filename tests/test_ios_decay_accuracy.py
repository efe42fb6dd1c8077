"""Accuracy of the intersection-over-self decay (a13, csrc/ios.cu) and the final ranking (a14) against exact counts and
float64 references, per element, on every path the product takes.

The stage's IoS reaches the golden comparisons only through the final scores, at 1e-3 of the image's largest score: a
count that is off by a few words in one of the evaluation branches still passes there.  These tests read the decay's
inputs through the taps of `nttt_match_args` (`sel`, `ios`, `ios_inter`, with `sim` and `obj_feats`) and check each
stage against a reference built from the kernel's own upstream outputs, so that a pooling or NMS difference cannot
leak in:
  inter64  exact same-label intersection counts of the selected masks.  The masks are rebuilt with the standalone
           `upsample_threshold_pack` + `unpack_masks` (pinned bit-exact to the C oracle) on the kernel's own `sel`, and
           multiplied per label group in fp32 with TF32 off, in slices of 2^18 pixels: every partial sum is an integer
           below 2^24, so the products are exact.
  ios64    the reference's formula max_{j != i, same label} ((inter_ij * s_ij) / area_i) * s_ij with
           s_ij = max(f_i . f_j, 0), in float64 from the obj_feats tap (compute_semantic_ios,
           matching_baseline_utils.py:831-867).  Rows without an intersecting partner are 0.

Checks on every stage case:
  1. counts: `ios_inter` equals inter64 exactly, zeros across labels and on the diagonal included;
  2. IoS values: |ios - ios64| <= TOL_IOS * bound_i per row, with the row's own bound
     bound_i = max_j (inter_ij / area_i) * (2 s_ij sum_k |f_ik f_jk| + s_ij^2): the first term carries the fp32 dot
     product's error through s^2, the second the three fp32 roundings of ((inter * s) / area) * s.  Area-0 rows are
     exactly 0 in the tap and NaN in the output; no selected row has a non-finite obj_feats row (the kernel clamps a
     NaN similarity to 0 where the reference would propagate it; such rows score NaN and are never selected);
  3. decay, bit for bit: d = f32(top) * sqrt(f32(1 - ios)) in numpy float32, top = the row maximum of the sim tap at
     sel[k]; the output scores are d[order], order is the stable argsort with NaN first and ties to the lower slot,
     out_index == sel[order], and labels, boxes and masks are those of the ranked slots;
  4. reachability: the branches a case is meant for are asserted from the geometry on the host (the pair kernel's
     word-window formula on the full-resolution boxes, the evaluation kernel's window clipped to the rects).

Tolerance.  TOL_IOS = 4e-7 is ~4x the largest normalised error measured on a B200 (1.02e-7, below).  It is also fine
enough that a count error shows in the float check on its own: a count off by one pixel moves row i by s^2 / area_i,
and RESOLUTION_PX = 1 asserts that TOL_IOS * bound_i stays below that in every row with an intersecting partner (the
`px` column below is the largest TOL_IOS * bound_i per case, in pixels of s^2 / area_i).  The reference's own fp32
values (golden `ios`, CPU sgemm for s) are held to TOL_REF_IOS = 1.2e-6, ~2x their largest error of 5.4e-7.

Measured on one B200 (1000 W power limit), largest normalised IoS error, throughput | low latency, and px:
  config2       7.7e-8 | 8.4e-8   px 0.20      v1_120x4096   8.2e-8 | 9.0e-8   px 0.30
  big_blobs     9.6e-8 | 9.1e-8   px 0.96      v1_200x180    7.4e-8 | 7.6e-8   px 0.008
  wide_2040     7.0e-8 | 7.4e-8   px 0.50      sel_2048      8.1e-8 | 8.2e-8   px 0.010
  v1_64x4096    8.2e-8 | 9.3e-8   px 0.031     sel_8192      1.02e-7 | 9.3e-8  px 0.002
  golden stage_* cases, both modes: <= 7.0e-8, px <= 0.17
  nttt_mask_ios: big_rowmajor 6.2e-8, wide_64x4096 4.3e-8, all_overlap 6.9e-8; the mixed 40-mask 333 x 500 case of
                 test_gpu_parity.py::test_mask_ios_counts_bit_exact 1.8e-8

Branches.  launch_upsample_pack runs the v2 resize (plan + work list, writing only the word-column-major copy `bits_t`)
when both axes have <= 3 taps (`tx.pk && ty.pk`), i.e. when the output is at least as large as the low-res masks on
both axes; IoS then reads `bits_t`.  Otherwise the v1 resize writes the row-major `bits_full` and IoS reads that.  In
throughput mode IoS runs ios_meta_kernel + ios_pairs_kernel; in low-latency mode after a v2 resize it runs
ios_pairs_fused_kernel, which relies on the resize having zeroed the pair counters (after a v1 resize both modes run
the unfused pair); ios_eval_kernel evaluates windows of <= 4096 words with one warp per pair and the rest in its
CTA-per-pair tail ios_eval_big_pairs.  decay_rank_kernel sorts n_pad = 1024 keys in registers and larger n_pad in the
shared-memory bitonic network, with dynamic shared memory above 4096 keys.
  config2       1024 masks, c 1024, 80 cls, 1024^2, clustered: v2, column-major warp eval (and its big tail), n_pad 1024
  big_blobs     one class, lr radii 80..160, nms 1.0, 1024^2: v2, big-pair tail in column-major, pair list >= 90% of
                ios_max_pairs
  wide_2040     1500 x 2040: v2 with 64-word rows
  v1_64x4096    64 x 4096: v1, row-major, warp windows wider than 32 words
  v1_120x4096   120 x 4096, big blobs, nms 1.0: v1, big-pair tail in row-major
  v1_200x180    200 x 180, degenerate masks: v1, empty full-res masks (ios 0 in the tap, NaN out)
  sel_2048      num_out 200, 2048 masks, nms 1.0: n_pad 2048, shared-memory network
  sel_8192      num_out 1024, 8192 masks of 64 x 64, 96 x 96 out, nms 1.0: v2, n_pad 8192, dynamic shared memory
Every case runs in throughput mode and in low-latency mode.  The golden stage_* cases run through the same checks, and
their rebuilt masks must hash to the golden `full_masks_sha`; a CPU test pins the float64 helper to the reference's
stored `ios` on the golden obj_feats and its counts to the C oracle.

Standalone entries: `nttt_mask_ios` (row-major, unfused, finalize: area-0 rows NaN) on the row-major big-pair tail,
windows wider than 32 words and one class whose pairs all overlap (test_gpu_parity.py::test_mask_ios_counts_bit_exact
runs the same checks on a small mixed case); `nttt_decay_topk` at max_sel 1024, 1025, 2048 and 8192 with crafted IoS
(exact ties, NaN, exactly 1, just above 1) and num_out above and below n_sel.
"""
import importlib

import numpy as np
import pytest
import torch

from golden_util import STAGE_CASES, load_case, sha_bool
from ios_ref import RESOLUTION_PX, TOL_IOS, TOL_REF_IOS, inter_counts, ios_errors, ios_reference
from oracle import nttt_oracle as orc

DEV = "cuda:0"

BIG_WORDS = 4096      # csrc/ios.cu kIosBigWords


def _synth():
    return importlib.import_module("no-time-to-train_b200.synth")


# ------------------------------------------------------------------------------------------------ references
def decay_order(top: np.ndarray, ios: np.ndarray):
    """-> (d, order): d = top * sqrt(1 - ios) in float32, and the stable descending order with NaN first (ties keep
    the lower slot), as torch.argsort(descending=True) on the reference's scores."""
    top = np.asarray(top, np.float32)
    with np.errstate(invalid="ignore"):
        d = top * np.sqrt(np.float32(1.0) - np.asarray(ios, np.float32))
    key = np.where(np.isnan(d), np.float32(np.inf), d)
    return d, np.argsort(-key, kind="stable")


def pair_geometry(box: torch.Tensor, rect: torch.Tensor, area: torch.Tensor, labels: torch.Tensor) -> dict:
    """The pair kernel's classification of the selected masks (same label, both non-empty, full-res boxes overlapping;
    big = window of ((x1 >> 5) - (x0 >> 5) + 1) * (y1 - y0 + 1) > 4096 words) and the evaluation kernel's word count of
    each window after clipping to both rects: -> counts of pairs, big pairs, and warp-path pairs wider than 32 words."""
    b, r = box.long(), rect.long()
    lab = labels.to(b.device).long()
    k = b.shape[0]
    x0 = torch.maximum(b[:, None, 0], b[None, :, 0])
    x1 = torch.minimum(b[:, None, 2], b[None, :, 2])
    y0 = torch.maximum(b[:, None, 1], b[None, :, 1])
    y1 = torch.minimum(b[:, None, 3], b[None, :, 3])
    upper = torch.ones((k, k), dtype=torch.bool, device=b.device).triu(1)
    live = area.to(b.device) > 0
    hit = upper & (lab[:, None] == lab[None, :]) & live[:, None] & live[None, :] & (x0 <= x1) & (y0 <= y1)
    big = hit & (((x1 >> 5) - (x0 >> 5) + 1) * (y1 - y0 + 1) > BIG_WORDS)
    wlo = torch.maximum(torch.maximum(r[:, None, 2], r[None, :, 2]), x0 >> 5)
    whi = torch.minimum(torch.minimum(r[:, None, 3], r[None, :, 3]), (x1 >> 5) + 1)
    wide = hit & ~big & (whi - wlo > 32)
    return dict(pairs=int(hit.sum()), big=int(big.sum()), wide=int(wide.sum()))


def resize_is_v2(lr_hw, ori_hw) -> bool:
    """launch_upsample_pack's condition `tx.pk && ty.pk`: <= 3 antialias taps on both axes (aa_max_taps:
    ceil(max(in / out, 1)) * 2 + 1), i.e. no down-scaling."""
    return all(np.float32(i) / np.float32(o) <= 1.0 for i, o in zip(lr_hw, ori_hw))


# ------------------------------------------------------------------------------------------------ CPU: golden
@pytest.mark.parametrize("name", STAGE_CASES)
def test_ios_reference_matches_golden(name):
    """The float64 helper, fed with the golden obj_feats, against the `ios` the real reference stored (fp32 products),
    within TOL_REF_IOS; its counts equal the C oracle's; the rebuilt masks hash to the golden full-res masks."""
    g, inp, cfg = load_case(name)
    sim = g["sim"]
    n = sim.shape[0]
    labels_all = sim.argmax(1)
    top = sim.max(1)
    if cfg["n_cls"] == 1:
        top = top * (top > top * np.float32(0.6))
    keep = g["nms_keep_full"][:min(8 * cfg["num_out_instance"], n)]
    sel = keep[top[keep] > 0]
    assert np.array_equal(labels_all[sel], g["labels_sel"])
    full = orc.aa_resize_threshold(inp.lr_masks.numpy()[sel], inp.ori_hw)
    assert sha_bool(full) == str(g["full_masks_sha"])
    area = full.reshape(len(sel), -1).sum(1)
    assert np.array_equal(area, g["full_area"])
    lab = torch.from_numpy(g["labels_sel"])
    inter = inter_counts(torch.from_numpy(full.astype(bool)), lab)
    f = g["obj_feats"][sel]
    _, o_inter = orc.semantic_ios(full, g["labels_sel"], np.maximum(f @ f.T, np.float32(0)), want_inter=True)
    assert np.array_equal(inter.numpy(), o_inter)
    ios64, bound, s2 = ios_reference(inter, torch.from_numpy(area), torch.from_numpy(f), lab)
    want = g["ios"].astype(np.float64)
    assert np.array_equal(np.isnan(want), area == 0), "the reference's NaN rows are its empty masks"
    err, px = ios_errors(torch.from_numpy(np.nan_to_num(want, nan=0.0)), ios64, bound, s2, name)
    print(f"[ios golden] {name}: reference ios err {err:.2e}, {int((area == 0).sum())} empty")
    assert err <= TOL_REF_IOS


def test_decay_order_semantics():
    """The ranking helper: NaN first (in slot order), then descending, ties to the lower slot; 1 - ios < 0 is NaN."""
    top = np.array([0.5, 0.25, 0.5, 0.9, 0.7, 0.5], np.float32)
    ios = np.array([0.75, 0.0, np.nan, 1.0, np.nextafter(np.float32(1), np.float32(2)), 0.75], np.float32)
    d, order = decay_order(top, ios)
    assert d[3] == 0.0 and np.isnan(d[2]) and np.isnan(d[4]) and d[0] == d[1] == d[5] == np.float32(0.25)
    assert order.tolist() == [2, 4, 0, 1, 5, 3]


# ------------------------------------------------------------------------------------------------ GPU: whole stage
# name: (n, c, n_cls, ori_hw, num_out, nms_thr, lr side, (rmin, rmax) at the low-res side, degenerate, expectations)
STAGE = {
    "config2": (1024, 1024, 80, (1024, 1024), 100, 0.5, 256, (4.0, 64.0), True, dict(v2=True)),
    "big_blobs": (1024, 256, 1, (1024, 1024), 100, 1.0, 256, (80.0, 160.0), False, dict(v2=True, big=True, full=0.9)),
    "wide_2040": (300, 256, 5, (1500, 2040), 100, 0.5, 256, (4.0, 64.0), True, dict(v2=True)),
    "v1_64x4096": (300, 256, 3, (64, 4096), 40, 0.7, 256, (16.0, 64.0), False, dict(v2=False, wide=True)),
    "v1_120x4096": (400, 256, 1, (120, 4096), 50, 1.0, 256, (48.0, 128.0), False, dict(v2=False, big=True)),
    "v1_200x180": (200, 384, 5, (200, 180), 100, 0.5, 256, (4.0, 64.0), True, dict(v2=False, empty=True)),
    "sel_2048": (2048, 256, 5, (256, 256), 200, 1.0, 256, (4.0, 64.0), False, dict(v2=True, n_pad=2048)),
    "sel_8192": (8192, 128, 16, (96, 96), 1024, 1.0, 64, (1.0, 16.0), False, dict(v2=True, n_pad=8192)),
}
MODES = ["throughput", "low_latency"]


def stage_inputs(name):
    n, c, n_cls, ori_hw, num_out, nms_thr, lr, (rmin, rmax), degenerate, _ = STAGE[name]
    synth = _synth()
    gen = torch.Generator().manual_seed(9000 + sorted(STAGE).index(name))
    masks = synth.make_masks(n, gen, lo=lr, rmin=rmin, rmax=rmax)
    pred_ious = 0.4 + 0.6 * torch.rand(n, generator=gen)
    feat, bank = synth.make_features(37 * 37, c, n_cls, 2, gen, clustered=True)
    if degenerate:
        synth.inject_degenerate_cases(masks, bank)
    return masks, pred_ious, feat, bank


_cases = {}


def _stage(P, name):
    """(stage, device inputs) of one case, cached while its modes run."""
    if name not in _cases:
        _cases.clear()
        torch.cuda.empty_cache()
        n, c, n_cls, ori_hw, num_out, nms_thr, *_ = STAGE[name]
        masks, ious, feat, bank = stage_inputs(name)
        stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=nms_thr, num_out_instance=num_out, enc_hw=(37, 37)))
        stage.set_prototypes(bank)
        _cases[name] = (stage, (masks.to(DEV), ious.to(DEV), feat.to(DEV), ori_hw))
    return _cases[name]


def check_stage(ops, out, lr_masks, ori_hw, n_cls, num_out, what, golden_sha=None):
    """Checks 1-3 of the module docstring on one `match(taps=True)` result -> (report dict, geometry)."""
    taps, counts = out["taps"], out["counts"]
    k = counts["n_sel"]
    max_sel = taps["sel"].shape[0]
    assert 0 < k <= max_sel, f"{what}: n_sel {k}"
    sel = taps["sel"][:k].contiguous()
    # the kernel's own upstream outputs: selection, features, similarities
    feats = taps["obj_feats"][sel.long()]
    assert torch.isfinite(feats).all(), f"{what}: a selected row has non-finite obj_feats"
    sim_sel = taps["sim"][sel.long()]
    top = sim_sel.max(dim=1).values
    if n_cls == 1:
        top = top * (top > top * 0.6)  # the reference's k == n_cls branch
    labels = sim_sel.argmax(dim=1)
    # the masks of the selection, rebuilt with the standalone entries
    bits, _, box, _, flags = ops.threshold_pack(lr_masks)
    n_sel = torch.tensor([k], dtype=torch.int32, device=DEV)
    bits_full, rect, area_full, box_full = ops.upsample_threshold_pack(lr_masks, bits, box, flags, sel, n_sel, k, ori_hw)
    masks = ops.unpack_masks(bits_full, rect, n_sel, ori_hw)
    if golden_sha is not None:
        assert sha_bool(masks) == golden_sha, f"{what}: rebuilt masks differ from the golden full-res masks"
    area = area_full[:k]
    # 1. counts
    inter = inter_counts(masks, labels)
    got_inter = taps["ios_inter"][:k, :k].to(torch.int64)
    bad = int((got_inter != inter).sum())
    assert bad == 0, f"{what}: {bad} intersection counts differ (largest |diff| {int((got_inter - inter).abs().max())})"
    if max_sel > k:
        assert not taps["ios_inter"][k:].any() and not taps["ios_inter"][:, k:].any(), f"{what}: counts past n_sel"
    # 2. IoS values
    ios64, bound, s2 = ios_reference(inter, area, feats, labels)
    ios_tap = taps["ios"][:k]
    empty = area == 0
    assert (ios_tap[empty] == 0).all(), f"{what}: an empty mask's row is not 0 in the tap"
    err, px = ios_errors(ios_tap, ios64, bound, s2, what)
    assert err <= TOL_IOS, f"{what}: normalised IoS error {err:.2e} > {TOL_IOS:.0e}"
    assert px <= RESOLUTION_PX, f"{what}: the tolerance spans {px:.2f} pixels of intersection"
    # 3. decay and ranking, bit for bit
    io = torch.where(empty, torch.full_like(ios_tap, float("nan")), ios_tap)
    d, order = decay_order(top.cpu().numpy(), io.cpu().numpy())
    n_out = min(num_out, k)
    order = order[:n_out]
    assert counts["n_out"] == n_out
    got_scores = out["scores"].cpu().numpy()
    assert np.array_equal(got_scores, d[order], equal_nan=True), f"{what}: decayed scores or their order differ"
    if empty.any():
        assert np.isnan(d[empty.cpu().numpy()]).all()
    o = torch.from_numpy(order).to(DEV)
    assert torch.equal(out["index"], sel[o]), f"{what}: out_index != sel[order]"
    assert torch.equal(out["labels"], labels[o]), f"{what}: labels"
    assert torch.equal(out["bboxes"], box_full[o].long()), f"{what}: boxes"
    assert torch.equal(out["binary_masks"], masks[o]), f"{what}: masks"
    geo = pair_geometry(box_full[:k], rect[:k], area, labels)
    rep = dict(n_sel=k, err=err, px=px, empty=int(empty.sum()), nan_out=int(np.isnan(got_scores).sum()), **geo,
               pairs_of_max=geo["pairs"] / (max_sel * (max_sel - 1) / 2 + 1))
    return rep


def _report(what, rep):
    print(f"[ios decay] {what} " + " ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}"
                                             for k, v in rep.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(STAGE))
def test_stage_ios_decay_per_element(ops, name, mode):
    """`MatchingStage.match(taps=True)`: counts exact, IoS per element, decay and ranking bit for bit, and the branch
    the case is meant for reached (module docstring)."""
    P = importlib.import_module("no-time-to-train_b200")
    n, c, n_cls, ori_hw, num_out, nms_thr, lr, _, _, expect = STAGE[name]
    stage, args = _stage(P, name)
    out = stage.match(*args, taps=True, low_latency=mode == "low_latency")
    rep = check_stage(ops, out, args[0], ori_hw, n_cls, num_out, f"{name} {mode}")
    _report(f"{name} {mode}", rep)
    assert resize_is_v2((lr, lr), ori_hw) == expect["v2"]
    max_sel = min(8 * num_out, n)
    if "n_pad" in expect:
        assert 1 << (max_sel - 1).bit_length() == expect["n_pad"]
    if expect.get("big"):
        assert rep["big"] > 0, f"{name}: no overlap window above {BIG_WORDS} words"
    if expect.get("wide"):
        assert rep["wide"] > 0, f"{name}: no warp-path window wider than 32 words"
    if expect.get("empty"):
        assert rep["empty"] > 0 and rep["nan_out"] > 0, f"{name}: no empty full-res mask reached the output"
    if "full" in expect:
        assert rep["pairs_of_max"] >= expect["full"], f"{name}: pair list {rep['pairs_of_max']:.2f} of ios_max_pairs"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", STAGE_CASES)
def test_stage_ios_decay_golden(ops, name, mode):
    """The golden stage cases through the same checks; the rebuilt masks are the reference's (golden hash)."""
    P = importlib.import_module("no-time-to-train_b200")
    g, inp, cfg = load_case(name)
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=cfg["num_out_instance"], enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    d = inp.lr_masks.to(DEV)
    out = stage.match(d, inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), inp.ori_hw, taps=True,
                      low_latency=mode == "low_latency")
    rep = check_stage(ops, out, d, inp.ori_hw, cfg["n_cls"], cfg["num_out_instance"], f"{name} {mode}",
                      golden_sha=str(g["full_masks_sha"]))
    assert rep["n_sel"] == len(g["labels_sel"])
    _report(f"{name} {mode}", rep)


# ------------------------------------------------------------------------------------------------ GPU: standalone
def _blob_masks(k, gen, centred=False, rmin=4.0, rmax=64.0):
    """`synth.make_masks` blobs, or (centred) blobs all around the same point, so that every pair overlaps."""
    if not centred:
        return _synth().make_masks(k, gen, rmin=rmin, rmax=rmax)
    ys = torch.arange(256, dtype=torch.float32).view(1, 256, 1)
    xs = torch.arange(256, dtype=torch.float32).view(1, 1, 256)
    r = 20.0 + 60.0 * torch.rand(k, 2, generator=gen)
    c = 128.0 + 10.0 * torch.randn(k, 2, generator=gen)
    dy = (ys - c[:, 0].view(k, 1, 1)) / r[:, 0].view(k, 1, 1)
    dx = (xs - c[:, 1].view(k, 1, 1)) / r[:, 1].view(k, 1, 1)
    return (8.0 * (1.0 - dy * dy - dx * dx) + 0.5 * torch.randn(k, 256, 256, generator=gen)).contiguous()


# name: (masks, ori_hw, n_cls, c, expectation, seed); the small mixed case is test_gpu_parity's
# test_mask_ios_counts_bit_exact
MASK_IOS = {
    "big_rowmajor": ((64, False, 48.0, 128.0), (1024, 1024), 1, 128, "big", 32),
    "wide_64x4096": ((96, False, 16.0, 64.0), (64, 4096), 2, 64, "wide", 34),
    "all_overlap": ((96, True, 0, 0), (480, 640), 1, 256, "all", 31),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MASK_IOS))
def test_mask_ios_per_element(ops, name):
    """`nttt_mask_ios` (row-major bits, unfused pairs, area-0 rows finalised to NaN): counts equal inter64 exactly,
    IoS per element against ios64."""
    (k, centred, rmin, rmax), ori_hw, n_cls, c, expect, seed = MASK_IOS[name]
    gen = torch.Generator().manual_seed(seed)
    logits = _blob_masks(k + 8, gen, centred, rmin, rmax)
    d = logits.to(DEV)
    bits, area, box, stab, flags = ops.threshold_pack(d)
    sel = torch.arange(k, dtype=torch.int32, device=DEV)
    n_sel = torch.tensor([k], dtype=torch.int32, device=DEV)
    bits_full, rect, area_full, box_full = ops.upsample_threshold_pack(d, bits, box, flags, sel, n_sel, k, ori_hw)
    labels = torch.randint(0, n_cls, (logits.shape[0],), generator=gen).int()
    feats = torch.nn.functional.normalize(torch.randn(logits.shape[0], c, generator=gen), dim=-1)
    if n_cls == 1:
        feats = torch.nn.functional.normalize(feats + 2.0 / c ** 0.5, dim=-1)  # mostly positive similarities
    ios, inter = ops.mask_ios(bits_full, rect, area_full, box_full, sel, n_sel, ori_hw, labels.to(DEV), feats.to(DEV),
                              want_inter=True)
    masks = ops.unpack_masks(bits_full, rect, n_sel, ori_hw)
    lab = labels[:k].to(DEV)
    want = inter_counts(masks, lab)
    assert torch.equal(inter.to(torch.int64), want), f"{name}: {int((inter.to(torch.int64) != want).sum())} counts differ"
    ios64, bound, s2 = ios_reference(want, area_full, feats[:k].to(DEV), lab)
    empty = area_full == 0
    assert torch.isnan(ios[empty]).all() and not torch.isnan(ios[~empty]).any()
    err, px = ios_errors(torch.where(empty, torch.zeros_like(ios), ios), ios64, bound, s2, name)
    geo = pair_geometry(box_full, rect, area_full, lab)
    _report(f"mask_ios {name}", dict(err=err, px=px, empty=int(empty.sum()), **geo))
    assert err <= TOL_IOS
    if expect == "big":
        assert geo["big"] > 0
    if expect == "wide":
        assert geo["wide"] > 0
    if expect == "all":
        live = int((~empty).sum())
        assert geo["pairs"] == live * (live - 1) // 2


@pytest.mark.gpu
@pytest.mark.parametrize("num_out", ["below", "above"])
@pytest.mark.parametrize("max_sel", [1024, 1025, 2048, 8192])
def test_decay_topk_crafted(ops, max_sel, num_out):
    """`nttt_decay_topk` on crafted IoS: exact ties (equal inputs, and different inputs with the same product), NaN,
    exactly 1 (score 0), just above 1 (sqrt of a negative: NaN, ranked first), an unused tail of the selection holding
    NaN; num_out below and above n_sel.  1024 runs the register sort, the others the shared-memory network (8192 with
    dynamic shared memory).  Scores, order, indices, slots, labels, boxes and masks bit for bit."""
    gen = torch.Generator().manual_seed(max_sel)
    n_src = max_sel + 7
    top = (0.05 + 0.9 * torch.rand(n_src, generator=gen)).float()
    sel = torch.randperm(n_src, generator=gen)[:max_sel].int()
    k = max_sel - 3
    ios = (0.9 * torch.rand(max_sel, generator=gen)).float()
    slots = torch.randperm(k, generator=gen)
    groups = slots[:64], slots[64:96], slots[96:112], slots[112:128], slots[128:144]
    top[sel[groups[0]].long()] = 0.5        # 0.5 * sqrt(1 - 0.75) = 0.25 exactly ...
    ios[groups[0]] = 0.75
    top[sel[groups[1]].long()] = 0.25       # ... = 0.25 * sqrt(1 - 0)
    ios[groups[1]] = 0.0
    ios[groups[2]] = float("nan")
    ios[groups[3]] = 1.0                    # score 0
    ios[groups[4]] = float(np.nextafter(np.float32(1), np.float32(2)))  # 1 - ios < 0: NaN
    ios[k:] = float("nan")                  # past n_sel: must not be read
    labels = torch.randint(0, 7, (n_src,), generator=gen).int()
    oh, ow = 3, 64
    bits_full = torch.randint(-2 ** 31, 2 ** 31 - 1, (max_sel, oh, ow // 32), generator=gen, dtype=torch.int64).int()
    rect = torch.tensor([0, oh, 0, ow // 32], dtype=torch.int32).repeat(max_sel, 1)
    box_full = torch.randint(0, 1000, (max_sel, 4), generator=gen).int()
    n_out_cap = k + 5 if num_out == "above" else 100
    dv = [t.to(DEV) for t in (top, labels, ios, sel, bits_full, rect, box_full)]
    n_sel = torch.tensor([k], dtype=torch.int32, device=DEV)
    masks, boxes, scores, out_labels, index, slot, n_out = ops.decay_topk(dv[0], dv[1], dv[2], dv[3], n_sel, n_out_cap,
                                                                          dv[4], dv[5], dv[6], (oh, ow))
    d, order = decay_order(top[sel[:k].long()].numpy(), ios[:k].numpy())
    m = min(n_out_cap, k)
    order = order[:m]
    assert int(n_out) == m
    assert np.isnan(d).sum() == 32 and (d == 0).sum() == 16 and (d == np.float32(0.25)).sum() >= 96
    assert np.array_equal(slot[:m].cpu().numpy(), order), "ranking order (NaN first, stable ties) differs"
    assert np.array_equal(scores[:m].cpu().numpy(), d[order], equal_nan=True)
    assert np.array_equal(index[:m].cpu().numpy(), sel.numpy()[order])
    assert np.array_equal(out_labels[:m].cpu().numpy(), labels.numpy()[sel.numpy()[order]])
    assert np.array_equal(boxes[:m].cpu().numpy(), box_full.numpy()[order])
    all_masks = ops.unpack_masks(dv[4], dv[5], n_sel, (oh, ow))
    assert torch.equal(masks[:m], all_masks[torch.from_numpy(order).to(DEV)])


@pytest.fixture(scope="module")
def ops():
    return importlib.import_module("no-time-to-train_b200.ops")
