"""One captured stage for images of any output size (`MatchingStage.graphed(..., min_hw=...)`, `nttt_match_image_sized`):
every replay at size (h, w) gives bit for bit what the eager stage gives at that size, the persistent mask buffer is the
dense result embedded top-left with zeros elsewhere, and a size outside the range gives an empty result and a status
without writing outside the capacity's buffers."""
import importlib

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (h, w) in a deliberately varying order: large after small and back, the capacity itself, widths that are not a
# multiple of 32 or 16, a size below the low-res 256 on both axes (general resize path), and a tall narrow one
SIZES = [(1024, 1024), (200, 180), (480, 640), (1024, 300), (333, 500), (640, 480), (256, 256), (427, 640),
         (640, 640)]


def _pkg():
    return importlib.import_module("no-time-to-train_b200")


def _inputs(seed, n=128, c=384, n_cls=9):
    P = _pkg()
    inp = P.synth.make_stage_inputs(n, c, n_cls, 2, (1, 1), seed=seed, clustered=True, degenerate=2)
    gen = torch.Generator().manual_seed(seed + 1)
    inp.pred_ious = torch.rand(n, generator=gen) * 0.6 + 0.4  # about a sixth fall below the 0.5 threshold
    inp.pred_ious[8:15] = 0.99  # the border cases reach the output
    return inp


def _stage(inp, num_out=20):
    P = _pkg()
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=num_out, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    return stage


def _load(g, inp):
    g.lr_masks.copy_(inp.lr_masks)
    g.pred_ious.copy_(inp.pred_ious)
    g.tar_feat.copy_(inp.tar_feat)


def _assert_same(out, eager, what):
    assert out["counts"] == eager["counts"], what
    assert torch.equal(torch.isnan(out["scores"]), torch.isnan(eager["scores"])), what
    assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(eager["scores"])), what
    assert torch.equal(out["labels"], eager["labels"]), what
    assert torch.equal(out["bboxes"], eager["bboxes"]), what
    assert torch.equal(out["index"], eager["index"]), what
    assert out["binary_masks"].shape == eager["binary_masks"].shape, what
    assert torch.equal(out["binary_masks"], eager["binary_masks"]), what


def _assert_embedded(full, eager_masks, what):
    """the WHOLE persistent buffer [num_out, H, W] == the eager masks in the top-left corner, zeros elsewhere"""
    want = torch.zeros_like(full)
    n, h, w = eager_masks.shape
    want[:n, :h, :w] = eager_masks
    assert torch.equal(full, want), what


@pytest.mark.parametrize("cap,min_hw,low_latency,rle", [
    ((1024, 1024), (256, 256), False, False),  # two-tap resize for every size of the range
    ((1024, 1024), (176, 160), False, True),   # both resize chains in one graph
    ((640, 640), (176, 160), True, True),
    ((640, 640), (256, 256), True, False),
])
def test_sizes_through_one_graph(cap, min_hw, low_latency, rle):
    inp = _inputs(301)
    stage = _stage(inp)
    g = stage.graphed(128, 384, cap, iou_thr=0.5, rle=rle, low_latency=low_latency, min_hw=min_hw).capture()
    sizes = [hw for hw in SIZES if min_hw[0] <= hw[0] <= cap[0] and min_hw[1] <= hw[1] <= cap[1]]
    assert cap in sizes and len(sizes) >= 6
    sizes = sizes + [sizes[1]]  # (the last replay lets nothing pass the filter)
    for step, hw in enumerate(sizes):
        cur = _inputs(310 + step)
        if step == len(sizes) - 1:
            cur.pred_ious[:] = 0.1
        _load(g, cur)
        pend = g.replay(ori_hw=hw)
        out = pend.get()
        eager = stage.match(cur.lr_masks.to(DEV), cur.pred_ious.to(DEV), cur.tar_feat.to(DEV), hw, iou_thr=0.5,
                            rle=rle, low_latency=low_latency)
        what = f"{hw} (step {step})"
        _assert_same(out, eager, what)
        assert (out["counts"]["n_out"] > 0) == (step != len(sizes) - 1), what
        _assert_embedded(g._out[0].view(torch.bool), eager["binary_masks"], what)
        if rle:
            segs = pend.rle_segmentations()
            assert segs == eager["segmentations"], what
            assert all(sg["size"] == [hw[0], hw[1]] for sg in segs), what


def test_back_to_back_replays_read_their_own_size():
    """Four replays of different sizes on one stream, no synchronisation in between: each result, copied out
    stream-ordered right behind its replay, is the eager result at its size — the size write of a replay never lands
    before the previous replay has read its own."""
    inp = _inputs(401)
    stage = _stage(inp)
    cap = (1024, 1024)
    g = stage.graphed(128, 384, cap, iou_thr=0.5, min_hw=(256, 256)).capture()
    sizes = [(1024, 300), (333, 500), (1024, 1024), (256, 256)]
    cases = [_inputs(410 + i) for i in range(len(sizes))]
    dev_in = [(c.lr_masks.to(DEV), c.pred_ious.to(DEV), c.tar_feat.to(DEV)) for c in cases]
    torch.cuda.synchronize()
    snaps = []
    for (lr, ious, feat), hw in zip(dev_in, sizes):
        g.lr_masks.copy_(lr)
        g.pred_ious.copy_(ious)
        g.tar_feat.copy_(feat)
        pend = g.replay(ori_hw=hw)
        snaps.append((hw, pend._meta_dev.clone(), g._out[0].clone(), pend.boxes.clone(), pend.scores.clone(),
                      pend.labels.clone(), pend.index.clone()))
    for (hw, meta, full, boxes, scores, labels, index), (lr, ious, feat) in zip(snaps, dev_in):
        eager = stage.match(lr, ious, feat, hw, iou_thr=0.5, low_latency=False)
        counts = meta.cpu().tolist()
        assert counts[3] == 0
        n_out = counts[2]
        assert dict(n_keep=counts[0], n_sel=counts[1], n_out=n_out) == eager["counts"], hw
        assert n_out > 0
        assert torch.equal(torch.nan_to_num(scores[:n_out]), torch.nan_to_num(eager["scores"])), hw
        assert torch.equal(labels[:n_out], eager["labels"]) and torch.equal(boxes[:n_out], eager["bboxes"]), hw
        assert torch.equal(index[:n_out], eager["index"]), hw
        _assert_embedded(full.view(torch.bool), eager["binary_masks"], hw)


def test_fused_multimask_selection_through_a_sized_graph():
    P = _pkg()
    n, m, c = 64, 4, 384
    inp = _inputs(501, n=n, c=c)
    stage = _stage(inp)
    g = stage.graphed(n, c, (640, 640), iou_thr=0.5, n_multi=m, min_hw=(256, 256)).capture()
    for seed, hw in ((502, (480, 640)), (503, (333, 500))):
        multi, ious = P.synth.make_multimask_inputs(n, m, seed=seed)
        feat = _inputs(seed, n=n, c=c).tar_feat
        g.lr_masks.copy_(multi)
        g.multi_ious.copy_(ious)
        g.tar_feat.copy_(feat)
        out = g.replay(ori_hw=hw).get()
        eager = stage.match(multi.to(DEV), None, feat.to(DEV), hw, iou_thr=0.5, multi_ious=ious.to(DEV),
                            multi_first=1, low_latency=False)
        assert eager["counts"]["n_out"] > 0
        _assert_same(out, eager, hw)
        _assert_embedded(g._out[0].view(torch.bool), eager["binary_masks"], hw)


def test_negative_reference_scoring_through_a_sized_graph():
    inp = _inputs(601)
    stage = _stage(inp)
    gen = torch.Generator().manual_seed(602)
    n_cls, l_neg, c = 9, 3, 384
    stage.set_prototypes_with_negatives(torch.randn(n_cls, c, generator=gen), torch.randn(n_cls, l_neg, c, generator=gen))
    g = stage.graphed(128, c, (1024, 1024), iou_thr=0.5, low_latency=True, min_hw=(200, 180)).capture()
    for seed, hw in ((603, (427, 640)), (604, (200, 180))):
        cur = _inputs(seed)
        _load(g, cur)
        out = g.replay(ori_hw=hw).get()
        eager = stage.match(cur.lr_masks.to(DEV), cur.pred_ious.to(DEV), cur.tar_feat.to(DEV), hw, iou_thr=0.5,
                            low_latency=True)
        assert eager["counts"]["n_out"] > 0
        _assert_same(out, eager, hw)


def test_replay_outside_the_range_raises_before_enqueueing():
    inp = _inputs(701)
    stage = _stage(inp)
    g = stage.graphed(128, 384, (640, 640), iou_thr=0.5, min_hw=(256, 256)).capture()
    _load(g, inp)
    g.replay(ori_hw=(480, 640)).get()
    for bad in ((255, 640), (480, 641), (641, 200), (100, 100)):
        with pytest.raises(ValueError, match="outside"):
            g.replay(ori_hw=bad)
    with pytest.raises(ValueError):
        g.replay()  # a sized graph needs the size
    assert g.hw_dev.cpu().tolist() == [480, 640]  # nothing was written
    static = stage.graphed(128, 384, (480, 640), iou_thr=0.5)
    with pytest.raises(ValueError):
        static.replay(ori_hw=(333, 500))


def _sized_call(stage, inp, cap, min_hw, hw, persistent):
    hw_dev = torch.tensor(hw, dtype=torch.int32, device=DEV)
    pend = stage.match_async(inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), cap, iou_thr=0.5,
                             persistent_out=persistent, size_range=(hw_dev, min_hw))
    pend.ori_hw = hw
    return pend


def test_device_size_outside_the_range_gives_an_empty_result():
    """Through the C entry: a size below the minimum, or above the capacity with output buffers that are really larger
    than the declared capacity, yields counts[3] != 0, an empty result, cleared persistent slots, and no byte written
    outside the declared capacity (the slack keeps its fill pattern)."""
    inp = _inputs(801)
    stage = _stage(inp, num_out=16)
    cap, min_hw = (480, 640), (256, 256)
    plane = cap[0] * cap[1]
    slack = 1 << 20
    raw = torch.full((16 * plane + slack,), 0xAB, dtype=torch.uint8, device=DEV)
    raw[:16 * plane].zero_()
    masks = raw[:16 * plane].view(16, cap[0], cap[1])
    prev = torch.zeros((16, 4), dtype=torch.int32, device=DEV)
    ok = _sized_call(stage, inp, cap, min_hw, (427, 640), (masks, prev)).get()
    assert ok["counts"]["n_out"] > 0 and bool(masks.any())
    for bad in ((200, 640), (480, 100), (481, 640), (480, 700), (4096, 4096), (0, 0), (-1, 640)):
        pend = _sized_call(stage, inp, cap, min_hw, bad, (masks, prev))
        counts = pend._meta_dev.cpu().tolist()
        assert counts[3] != 0 and counts[1] == 0 and counts[2] == 0, bad
        with pytest.raises(RuntimeError, match="outside"):
            pend.get()
        assert not bool(masks.any()), f"{bad}: persistent slots not cleared"
        assert bool((raw[16 * plane:] == 0xAB).all()), f"{bad}: bytes written beyond the capacity"
        assert not bool(prev.any()), bad
    # and a valid size afterwards is served normally again
    again = _sized_call(stage, inp, cap, min_hw, (427, 640), (masks, prev))
    out = again.get()
    eager = stage.match(inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), (427, 640), iou_thr=0.5,
                        low_latency=False)
    _assert_same(out, eager, "after the out-of-range calls")
    assert again._meta_dev.cpu().tolist()[3] == 0
    stats = stage.atlas_stats()
    assert stats["atlases"] >= 1 and stats["bytes"] > 0
