"""A captured stage with its inputs bound at replay (`MatchingStage.graphed(..., bind=True)`, `nttt_match_bind`,
`nttt_match_image_bound`): every replay on a producer's own tensors, at addresses the capture never saw, gives bit for
bit what the eager stage gives on the same tensors.  Also: graphs re-capture after the stage's prototypes are replaced,
and malformed inputs are rejected on the host before anything is enqueued."""
import importlib

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pkg():
    return importlib.import_module("no-time-to-train_b200")


def _inputs(seed, n=128, c=384, n_cls=9):
    P = _pkg()
    inp = P.synth.make_stage_inputs(n, c, n_cls, 2, (1, 1), seed=seed, clustered=True, degenerate=2)
    gen = torch.Generator().manual_seed(seed + 1)
    inp.pred_ious = torch.rand(n, generator=gen) * 0.6 + 0.4  # about a sixth fall below the 0.5 threshold
    inp.pred_ious[8:15] = 0.99  # the border cases reach the output
    return inp


def _dev(inp):
    """fresh device copies: addresses the graph's capture never saw"""
    return inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV)


def _stage(inp, num_out=20):
    P = _pkg()
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=num_out, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    return stage


def _assert_same(out, eager, what):
    assert out["counts"] == eager["counts"], what
    assert torch.equal(torch.isnan(out["scores"]), torch.isnan(eager["scores"])), what
    assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(eager["scores"])), what
    assert torch.equal(out["labels"], eager["labels"]), what
    assert torch.equal(out["bboxes"], eager["bboxes"]), what
    assert torch.equal(out["index"], eager["index"]), what
    assert out["binary_masks"].shape == eager["binary_masks"].shape, what
    assert torch.equal(out["binary_masks"], eager["binary_masks"]), what


@pytest.mark.parametrize("low_latency", [False, True])
def test_one_bound_graph_serves_many_input_sets(low_latency):
    inp = _inputs(101)
    stage = _stage(inp)
    hw = (480, 640)
    g = stage.graphed(128, 384, hw, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True).capture()
    static = {g.lr_masks.data_ptr(), g.pred_ious.data_ptr(), g.tar_feat.data_ptr()}
    held, nan_seen = [], False
    for step in range(7):
        cur = _inputs(110 + step)
        if step == 6:
            cur.pred_ious[:] = 0.1  # nothing passes the filter
        lr, ious, feat = _dev(cur)
        held.append((lr, ious, feat))
        assert not static & {lr.data_ptr(), ious.data_ptr(), feat.data_ptr()}
        pend = g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)
        out = pend.get()
        eager = stage.match(lr, ious, feat, hw, iou_thr=0.5, rle=True, low_latency=low_latency)
        what = f"step {step}"
        _assert_same(out, eager, what)
        assert (out["counts"]["n_out"] > 0) == (step != 6), what
        assert pend.rle_segmentations() == eager["segmentations"], what
        nan_seen |= bool(torch.isnan(out["scores"]).any())
    assert nan_seen  # (the degenerate masks reach the output: the NaN pattern was compared)


def test_fused_multimask_from_the_decoders_chunk_list():
    P = _pkg()
    n, m, c, cp = 64, 4, 384, 24  # chunks of 24, 24 and 16 prompts
    stage = _stage(_inputs(201, n=n, c=c))
    hw = (427, 640)
    g = stage.graphed(n, c, hw, iou_thr=0.5, n_multi=m, bind=True, chunk_prompts=cp).capture()
    assert [t.shape[0] for t in g.lr_masks] == [24, 24, 16]
    for seed in (202, 203, 204):
        multi, ious = P.synth.make_multimask_inputs(n, m, seed=seed)
        chunks = [t.to(DEV) for t in multi.split(cp)]  # separate allocations, as the decoder returns them
        ious, feat = ious.to(DEV), _inputs(seed, n=n, c=c).tar_feat.to(DEV)
        out = g.replay(lr_masks=chunks, multi_ious=ious, tar_feat=feat).get()
        eager = stage.match(chunks, None, feat, hw, iou_thr=0.5, multi_ious=ious, multi_first=1, low_latency=False)
        assert eager["counts"]["n_out"] > 0
        _assert_same(out, eager, seed)


def test_sized_bound_graph_serves_several_sizes():
    inp = _inputs(301)
    stage = _stage(inp)
    cap = (1024, 1024)
    g = stage.graphed(128, 384, cap, iou_thr=0.5, min_hw=(176, 160), bind=True).capture()
    for step, hw in enumerate([(1024, 1024), (200, 180), (480, 640), (1024, 300), (333, 500)]):
        lr, ious, feat = _dev(_inputs(310 + step))
        out = g.replay(ori_hw=hw, lr_masks=lr, pred_ious=ious, tar_feat=feat).get()
        eager = stage.match(lr, ious, feat, hw, iou_thr=0.5, low_latency=False)
        _assert_same(out, eager, hw)
        assert out["counts"]["n_out"] > 0
        want = torch.zeros_like(g._out[0].view(torch.bool))
        k, h, w = eager["binary_masks"].shape
        want[:k, :h, :w] = eager["binary_masks"]
        assert torch.equal(g._out[0].view(torch.bool), want), hw  # the dense result embedded, zeros elsewhere
        assert g.hw_dev.cpu().tolist() == list(hw)


def test_negative_reference_scoring_through_a_bound_graph():
    inp = _inputs(401)
    stage = _stage(inp)
    gen = torch.Generator().manual_seed(402)
    n_cls, l_neg, c = 9, 3, 384
    stage.set_prototypes_with_negatives(torch.randn(n_cls, c, generator=gen), torch.randn(n_cls, l_neg, c, generator=gen))
    g = stage.graphed(128, c, (640, 640), iou_thr=0.5, low_latency=True, bind=True).capture()
    for seed in (403, 404):
        lr, ious, feat = _dev(_inputs(seed))
        out = g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat).get()
        eager = stage.match(lr, ious, feat, (640, 640), iou_thr=0.5, low_latency=True)
        assert eager["counts"]["n_out"] > 0
        _assert_same(out, eager, seed)


def test_bound_replays_alternate_with_replays_on_the_static_buffers():
    inp = _inputs(501)
    stage = _stage(inp)
    hw = (640, 480)
    g = stage.graphed(128, 384, hw, iou_thr=0.5, bind=True).capture()
    for step in range(3):
        own = _inputs(510 + step)
        g.lr_masks.copy_(own.lr_masks)
        g.pred_ious.copy_(own.pred_ious)
        g.tar_feat.copy_(own.tar_feat)
        out = g.replay().get()
        eager = stage.match(g.lr_masks, g.pred_ious, g.tar_feat, hw, iou_thr=0.5, low_latency=False)
        _assert_same(out, eager, f"static {step}")
        lr, ious, feat = _dev(_inputs(520 + step))
        out = g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat).get()
        eager = stage.match(lr, ious, feat, hw, iou_thr=0.5, low_latency=False)
        _assert_same(out, eager, f"bound {step}")
        # only the features bound: the masks and scores are the static buffers'
        out = g.replay(tar_feat=feat).get()
        eager = stage.match(g.lr_masks, g.pred_ious, feat, hw, iou_thr=0.5, low_latency=False)
        _assert_same(out, eager, f"partly bound {step}")


@pytest.mark.parametrize("bind", [False, True])
def test_prototypes_replaced_after_capture(bind):
    """A graph reads the prototypes' address; replacing them re-captures on the next replay, and the old tensors stay
    alive until then."""
    inp = _inputs(601)
    stage = _stage(inp)
    hw = (480, 640)
    g = stage.graphed(128, 384, hw, iou_thr=0.5, bind=bind).capture()
    lr, ious, feat = _dev(inp)
    g.lr_masks.copy_(lr)
    g.pred_ious.copy_(ious)
    g.tar_feat.copy_(feat)
    before = g.replay().get()
    _assert_same(before, stage.match(lr, ious, feat, hw, iou_thr=0.5, low_latency=False), "first bank")
    gen = torch.Generator().manual_seed(602)
    for bank in range(2):
        stage.set_prototypes(inp.feats_ins_avg[torch.randperm(inp.feats_ins_avg.shape[0], generator=gen)] +
                             0.05 * torch.randn(inp.feats_ins_avg.shape, generator=gen))
        torch.empty(stage.proto.numel() * 4, device=DEV).fill_(float("nan"))  # (reuses freed memory, if any)
        out = g.replay().get()
        eager = stage.match(lr, ious, feat, hw, iou_thr=0.5, low_latency=False)
        if bank == 0:
            assert not torch.equal(eager["labels"], before["labels"])  # (the bank decides the result)
        _assert_same(out, eager, f"bank {bank}")


def test_malformed_inputs_raise_before_enqueueing():
    inp = _inputs(701)
    stage = _stage(inp)
    hw = (480, 640)
    g = stage.graphed(128, 384, hw, iou_thr=0.5, bind=True).capture()
    lr, ious, feat = _dev(inp)
    good = g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat).get()
    struct = g.inputs_dev.clone()
    offset = torch.empty(lr.numel() + 1, device=DEV)[1:].view_as(lr)
    offset.copy_(lr)
    bad = [
        dict(lr_masks=lr.double()),                            # dtype
        dict(pred_ious=ious.half()),
        dict(lr_masks=lr[:100]),                               # shape
        dict(tar_feat=feat[:, :256].contiguous()),
        dict(pred_ious=ious.cpu()),                            # device
        dict(tar_feat=feat.t().contiguous().t()),              # not contiguous
        dict(lr_masks=lr.transpose(1, 2)),
        dict(lr_masks=offset),                                 # 4 bytes off the 16-byte boundary
        dict(multi_ious=torch.zeros(128, 4, device=DEV)),      # not this graph's kind of input
    ]
    for kw in bad:
        with pytest.raises((TypeError, ValueError)):
            g.replay(lr_masks=kw.get("lr_masks", lr), pred_ious=kw.get("pred_ious", ious),
                     tar_feat=kw.get("tar_feat", feat), multi_ious=kw.get("multi_ious"))
    torch.cuda.synchronize()
    assert torch.equal(g.inputs_dev, struct)  # nothing was bound
    static = stage.graphed(128, 384, hw, iou_thr=0.5)
    with pytest.raises(ValueError, match="bind=True"):
        static.replay(lr_masks=lr)
    assert static.graph is None  # (nothing captured either)
    # chunk lists: count and per-chunk shape
    P = _pkg()
    mg = stage.graphed(64, 384, hw, iou_thr=0.5, n_multi=4, bind=True, chunk_prompts=24)
    multi, mious = P.synth.make_multimask_inputs(64, 4, seed=702)
    chunks = [t.to(DEV) for t in multi.split(24)]
    mious, mfeat = mious.to(DEV), feat
    for wrong in (chunks[:2], chunks + [chunks[-1]], [chunks[0], chunks[2], chunks[1]], torch.cat(chunks)):
        with pytest.raises(ValueError):
            mg.replay(lr_masks=wrong, multi_ious=mious, tar_feat=mfeat)
    assert mg.graph is None
    out = mg.replay(lr_masks=chunks, multi_ious=mious, tar_feat=mfeat).get()
    eager = stage.match(chunks, None, mfeat, hw, iou_thr=0.5, multi_ious=mious, multi_first=1, low_latency=False)
    _assert_same(out, eager, "chunks after the rejections")
    assert good["counts"]["n_out"] > 0
