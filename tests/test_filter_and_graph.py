"""Fused candidate filter (`scores_all > iou_thr`, Sam2MatchingBaseline_noAMG.py:428-431) and CUDA-graph replay of
the whole stage: both must give exactly what the reference gives on the compacted inputs."""
import importlib

import numpy as np
import pytest
import torch

from golden_util import assert_rows_match, assert_same_ranking
from oracle import ref_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _case(n=96, c=256, n_cls=6, seed=61, ori_hw=(384, 512)):
    P = importlib.import_module("no-time-to-train_b200")
    inp = P.synth.make_stage_inputs(n, c, n_cls, 2, ori_hw, seed=seed, clustered=True, degenerate=True)
    gen = torch.Generator().manual_seed(seed + 1)
    inp.pred_ious = torch.rand(n, generator=gen)  # about 40 % fall below the 0.4 threshold
    inp.pred_ious[5] = 0.4                        # exactly the threshold: dropped (strict >)
    return P, inp


def test_fused_iou_filter_equals_compaction():
    P, inp = _case()
    thr = 0.4
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=12, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    got = stage.match(inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), inp.ori_hw, iou_thr=thr)
    keep = inp.pred_ious > thr
    assert 10 < int(keep.sum()) < inp.lr_masks.shape[0] - 10
    # the reference semantics: compact first, then run the stage
    ref = ref_torch.match_image(inp.lr_masks[keep], inp.pred_ious[keep], inp.tar_feat, inp.feats_ins_avg,
                                ref_torch.StageConfig(num_out_instance=12), inp.ori_hw)
    assert got["counts"]["n_keep"] == ref["aux"]["keep"].numel()
    assert got["counts"]["n_sel"] == ref["aux"]["sel_index"].numel()
    assert_same_ranking(got["scores"].cpu().numpy(), got["labels"].cpu().numpy(), ref["scores"].numpy(),
                        ref["labels"].numpy(), what="filtered")
    # our indices refer to the un-compacted list
    orig_index = torch.nonzero(keep).flatten()[ref["aux"]["sel_index"][ref["aux"]["order"]]]
    assert_rows_match(dict(scores=got["scores"], labels=got["labels"], bboxes=got["bboxes"], masks=got["binary_masks"],
                           index=got["index"]),
                      dict(scores=ref["scores"], labels=ref["labels"], bboxes=ref["bboxes"], masks=ref["binary_masks"],
                           index=orig_index), what="filtered")
    # and the same through the compacted call of our own stage
    own = stage.match(inp.lr_masks[keep].contiguous().to(DEV), inp.pred_ious[keep].contiguous().to(DEV),
                      inp.tar_feat.to(DEV), inp.ori_hw)
    assert torch.equal(torch.nan_to_num(own["scores"]), torch.nan_to_num(got["scores"]))
    assert torch.equal(own["binary_masks"], got["binary_masks"])


def test_filter_everything_gives_empty_result():
    P, inp = _case(n=32)
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=5, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    got = stage.match(inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), inp.ori_hw, iou_thr=2.0)
    assert got["counts"]["n_keep"] == 0 and got["binary_masks"].shape[0] == 0


def test_graph_replay_matches_eager():
    P, inp = _case(n=128, c=384, n_cls=9, seed=71, ori_hw=(1024, 1024))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=20, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    g = stage.graphed(128, 384, (1024, 1024), iou_thr=0.4).capture()
    for seed in (71, 72, 73):  # new inputs written into the static buffers, same graph
        _, cur = _case(n=128, c=384, n_cls=9, seed=seed, ori_hw=(1024, 1024))
        g.lr_masks.copy_(cur.lr_masks)
        g.pred_ious.copy_(cur.pred_ious)
        g.tar_feat.copy_(cur.tar_feat)
        out = g.replay().get()
        eager = stage.match(cur.lr_masks.to(DEV), cur.pred_ious.to(DEV), cur.tar_feat.to(DEV), (1024, 1024), iou_thr=0.4,
                            low_latency=False)  # same accumulation order as the captured (throughput-mode) graph
        assert out["counts"] == eager["counts"]
        assert torch.equal(torch.isnan(out["scores"]), torch.isnan(eager["scores"]))
        assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(eager["scores"]))
        assert torch.equal(out["labels"], eager["labels"])
        assert torch.equal(out["binary_masks"], eager["binary_masks"]) and torch.equal(out["bboxes"], eager["bboxes"])


def test_low_latency_graph_replay_matches_eager():
    """The low-latency launch mode under stream capture: the side-stream fork (feature / prototype operand preparation)
    and the programmatic dependent launches along the kernel chain become graph edges.  Every replay — new inputs in the
    static buffers, several replays back to back without a host synchronisation in between — gives bit for bit what
    the eager low-latency call gives, with RLE output and persistent masks."""
    P, inp = _case(n=128, c=384, n_cls=9, seed=171, ori_hw=(640, 480))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=20, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    g = stage.graphed(128, 384, (640, 480), iou_thr=0.4, rle=True, low_latency=True).capture()
    for seed in (171, 172, 173, 174):
        _, cur = _case(n=128, c=384, n_cls=9, seed=seed, ori_hw=(640, 480))
        g.lr_masks.copy_(cur.lr_masks)
        g.pred_ious.copy_(cur.pred_ious)
        g.tar_feat.copy_(cur.tar_feat)
        for _ in range(3):  # the same image three times: a replay must not depend on what the previous one left behind
            pend = g.replay()
        out = pend.get()
        segs = pend.rle_segmentations()
        eager = stage.match(cur.lr_masks.to(DEV), cur.pred_ious.to(DEV), cur.tar_feat.to(DEV), (640, 480), iou_thr=0.4,
                            rle=True, low_latency=True)
        assert out["counts"] == eager["counts"]
        assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(eager["scores"]))
        assert torch.equal(out["labels"], eager["labels"]) and torch.equal(out["bboxes"], eager["bboxes"])
        assert torch.equal(out["binary_masks"], eager["binary_masks"])
        assert segs == eager["segmentations"]


def test_low_latency_chain_is_deterministic_over_many_calls():
    """Race check of the overlapped kernel chain (programmatic dependent launch: a kernel may be scheduled while its
    predecessor is finishing, and waits for it before its first read): 60 back-to-back calls on two alternating images
    give the same bits every time, and the taps written by the middle of the chain as well."""
    P, a = _case(n=192, c=384, n_cls=9, seed=181, ori_hw=(512, 768))
    _, b = _case(n=192, c=384, n_cls=9, seed=182, ori_hw=(512, 768))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=30, enc_hw=(37, 37)))
    stage.set_prototypes(a.feats_ins_avg)
    dev_in = [(x.lr_masks.to(DEV), x.pred_ious.to(DEV), x.tar_feat.to(DEV)) for x in (a, b)]
    first = [None, None]
    for rep in range(60):
        pend = stage.match_async(*dev_in[rep % 2], (512, 768), taps=True, iou_thr=0.3, low_latency=True)
        if rep % 7 == 3:
            torch.cuda.synchronize()  # (some calls start on an idle device, most behind the previous image's tail)
        out = pend.get()
        cur = (out["counts"], out["scores"].clone(), out["labels"].clone(), out["bboxes"].clone(),
               out["binary_masks"].clone(), out["taps"]["sim"].clone(), out["taps"]["obj_feats"].clone())
        if first[rep % 2] is None:
            first[rep % 2] = cur
            continue
        ref = first[rep % 2]
        assert cur[0] == ref[0], rep
        for x, y in zip(cur[1:], ref[1:]):
            assert torch.equal(torch.nan_to_num(x.float()), torch.nan_to_num(y.float())), rep


@pytest.mark.parametrize("n,c,ori_hw", [(300, 384, (480, 640)), (1000, 1024, (512, 512)), (130, 768, (333, 500))])
def test_pool_order_skips_only_zeros(n, c, ori_hw):
    """Throughput mode orders the rows of the pooling GEMM spatially and skips the k-blocks a tile of masks does not
    touch.  Skipped blocks are exact zeros: with the order switched off (`pool_order` 0) every output is bit-identical
    — pooled features and similarities included — and the low-latency mode (no order, split-K) agrees on every integer."""
    P, inp = _case(n=n, c=c, n_cls=9, seed=191, ori_hw=ori_hw)
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=40, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    args = (inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), inp.ori_hw)
    a = stage.match(*args, taps=True, low_latency=False)
    try:
        stage.tune("pool_order", 0)
        b = stage.match(*args, taps=True, low_latency=False)
    finally:
        stage.tune("pool_order", 1)
    ll = stage.match(*args, taps=True, low_latency=True)
    assert a["counts"] == b["counts"] == ll["counts"] and a["counts"]["n_out"] > 0
    for key in ("binary_masks", "bboxes", "labels"):
        assert torch.equal(a[key], b[key]) and torch.equal(a[key], ll[key]), key
    assert torch.equal(torch.nan_to_num(a["scores"]), torch.nan_to_num(b["scores"]))
    # (sign of an exact zero may differ: a skipped block adds nothing, a multiplied one may add -0.0)
    assert torch.equal(a["taps"]["obj_feats"] + 0.0, b["taps"]["obj_feats"] + 0.0)
    assert torch.equal(a["taps"]["sim"] + 0.0, b["taps"]["sim"] + 0.0)
    assert torch.allclose(a["taps"]["obj_feats"], ll["taps"]["obj_feats"], rtol=0, atol=1e-6)


def test_pool_order_keeps_nonfinite_features():
    """0 * inf = NaN in the reference's dense product: a k-block whose features hold an inf or a NaN is multiplied even
    where the masks' projections are all zero — same NaN pattern with and without the skipping."""
    P, inp = _case(n=300, c=384, n_cls=9, seed=192, ori_hw=(256, 256))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=40, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    feat = inp.tar_feat.clone()
    feat[5, 17] = float("inf")       # first encoder row, channel 17
    feat[1300, 200] = float("nan")   # last encoder rows, channel 200
    args = (inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), feat.to(DEV), inp.ori_hw)
    a = stage.match(*args, taps=True, low_latency=False)
    try:
        stage.tune("pool_order", 0)
        b = stage.match(*args, taps=True, low_latency=False)
    finally:
        stage.tune("pool_order", 1)
    fa, fb = a["taps"]["obj_feats"], b["taps"]["obj_feats"]
    assert bool(torch.isnan(fb).any())
    assert torch.equal(torch.isnan(fa), torch.isnan(fb))
    assert torch.equal(torch.nan_to_num(fa) + 0.0, torch.nan_to_num(fb) + 0.0)
    assert a["counts"] == b["counts"]


def test_persistent_outputs_are_exactly_the_dense_unpack():
    """Sparse unpack into persistent buffers: after every replay the WHOLE mask buffer (used and unused slots)
    equals what a dense unpack into a fresh buffer gives, also when the number of outputs shrinks to zero."""
    P, inp = _case(n=128, c=384, n_cls=9, seed=81, ori_hw=(480, 640))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=16, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    g = stage.graphed(128, 384, (480, 640), iou_thr=0.4).capture()
    for step, seed in enumerate((81, 82, 83, 84)):
        _, cur = _case(n=128, c=384, n_cls=9, seed=seed, ori_hw=(480, 640))
        if step == 2:
            cur.pred_ious[:] = 0.1  # nothing passes the filter: every slot must be cleared
        if step == 3:
            cur.pred_ious[8:] = 0.1  # only a handful of candidates
        g.lr_masks.copy_(cur.lr_masks)
        g.pred_ious.copy_(cur.pred_ious)
        g.tar_feat.copy_(cur.tar_feat)
        out = g.replay().get()
        eager = stage.match(cur.lr_masks.to(DEV), cur.pred_ious.to(DEV), cur.tar_feat.to(DEV), (480, 640), iou_thr=0.4,
                            low_latency=False)  # same accumulation order as the captured (throughput-mode) graph
        n_out = out["counts"]["n_out"]
        assert n_out == eager["counts"]["n_out"]
        full = g._out[0].view(torch.bool)
        assert torch.equal(full[:n_out], eager["binary_masks"])
        assert not bool(full[n_out:].any()), "stale pixels left in unused output slots"
    assert step == 3


def test_low_latency_mode_changes_no_integer_result():
    """`low_latency` only reshapes kernels (the pooling GEMM runs split-K): masks, boxes, labels and counts are
    identical, float scores agree to the last few bits."""
    P, inp = _case(n=128, c=384, n_cls=9, seed=91, ori_hw=(480, 640))
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=20, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    args = (inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV), inp.ori_hw)
    a = stage.match(*args, taps=True, low_latency=True)
    b = stage.match(*args, taps=True, low_latency=False)
    assert a["counts"] == b["counts"]
    assert torch.equal(a["binary_masks"], b["binary_masks"]) and torch.equal(a["bboxes"], b["bboxes"])
    assert torch.equal(a["labels"], b["labels"])
    assert torch.allclose(a["taps"]["obj_feats"], b["taps"]["obj_feats"], rtol=0, atol=1e-6)
    assert torch.allclose(torch.nan_to_num(a["scores"]), torch.nan_to_num(b["scores"]), rtol=1e-5, atol=1e-7)
