"""A captured stage with its candidate count bound at replay (`MatchingStage.graphed(..., counted=True)`,
`nttt_match_count_bind`, `nttt_match_image_counted`): one capture of capacity N serves compacted candidate lists of any
length k <= N.  Every replay gives bit for bit what the eager stage (`nttt_match_image`) gives on the k-row tensors, in
both launch modes: across the pooling-order threshold (128), the power-of-two edges, the NMS register / class-order
boundary (1024) and the split-K choices of the low-latency mode.  Rows past k are never read (poisoned rows change
nothing), a smaller count after a larger one sees no stale row, and k = 0 clears the persistent outputs.  A count outside
the capacity written straight to the device gives an empty result and the count status, and writes nothing outside the
buffers."""
import importlib

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
C = 1024  # DINOv2-L: the vector normalisation path and the spatially ordered pooling GEMM apply
HW = (480, 640)
MODES = [False, True]  # low_latency


def _pkg():
    return importlib.import_module("no-time-to-train_b200")


_CENTRES = {}


def _centres():
    if "c" not in _CENTRES:
        _CENTRES["c"] = _pkg().synth.cluster_centres(C)
    return _CENTRES["c"]


def _inputs(n, seed):
    lr, ious, feat = _pkg().synth.make_stage_inputs_device(n, _centres(), DEV, seed=seed)
    return lr, ious, feat


def _stage(num_out=20, n_cls=80):
    P = _pkg()
    st = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=num_out, enc_hw=(37, 37)))
    gen = torch.Generator().manual_seed(6)
    cen = _centres()
    st.set_prototypes((cen[torch.arange(n_cls) % cen.shape[0]] + 0.05 * torch.randn(n_cls, C, generator=gen)).unsqueeze(1))
    return st


def _poisoned(lr, ious, cap):
    """[cap] buffers whose rows past the live ones hold NaN / inf logits and NaN IoUs"""
    k = lr.shape[0]
    big_lr = torch.empty((cap, 256, 256), dtype=torch.float32, device=DEV)
    big_iou = torch.empty((cap,), dtype=torch.float32, device=DEV)
    big_lr[:k], big_iou[:k] = lr, ious
    big_lr[k:] = float("nan")
    big_lr[k::2] = float("inf")
    big_iou[k:] = float("nan")
    return big_lr, big_iou


def _eager(stage, lr, ious, feat, low_latency, hw=HW, iou_thr=None, taps=False, **kw):
    pend = stage.match_async(lr, ious, feat, hw, iou_thr=iou_thr, rle=True, low_latency=low_latency, taps=taps, **kw)
    out = pend.get()
    out["segmentations"] = pend.rle_segmentations()
    return out


def _replay(g, **kw):
    pend = g.replay(**kw)
    out = pend.get()
    out["segmentations"] = pend.rle_segmentations()
    return out


def _assert_same(out, ref, what):
    assert out["counts"] == ref["counts"], what
    assert torch.equal(torch.isnan(out["scores"]), torch.isnan(ref["scores"])), what
    assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(ref["scores"])), what
    assert torch.equal(out["labels"], ref["labels"]), what
    assert torch.equal(out["bboxes"], ref["bboxes"]), what
    assert torch.equal(out["index"], ref["index"]), what
    assert out["binary_masks"].shape == ref["binary_masks"].shape, what
    assert torch.equal(out["binary_masks"], ref["binary_masks"]), what
    assert out["segmentations"] == ref["segmentations"], what


def _assert_empty(out, g):
    assert out["counts"] == dict(n_keep=0, n_sel=0, n_out=0)
    assert out["segmentations"] == []
    assert int(g._out[0].count_nonzero()) == 0 and int(g._out[1].count_nonzero()) == 0  # persistent slots cleared


@pytest.mark.parametrize("low_latency", MODES)
def test_capacity_256_graph_serves_every_count(low_latency):
    """bound inputs: k-row views of [256] buffers poisoned past k; descending counts in a row, then 0, then growth"""
    cap = 256
    stage = _stage()
    lr, ious, feat = _inputs(cap, seed=11)
    g = stage.graphed(cap, C, HW, rle=True, low_latency=low_latency, bind=True, counted=True)
    graph = None
    for k in [256, 255, 129, 128, 7, 1, 0, 129, 256]:
        big_lr, big_iou = _poisoned(lr[:k], ious[:k], cap)
        out = _replay(g, lr_masks=big_lr[:k], pred_ious=big_iou[:k], tar_feat=feat)
        graph = graph or g.graph
        assert g.graph is graph  # (one capture serves every count)
        if k == 0:
            _assert_empty(out, g)
            continue
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency)
        _assert_same(out, ref, f"k={k}")
        assert out["counts"]["n_out"] > 0


@pytest.mark.parametrize("low_latency", MODES)
def test_capacity_2048_unbound_graph_across_the_nms_and_split_boundaries(low_latency):
    """static buffers poisoned past k, replay(n=k): 1000 and 1024 take the register NMS and 1025 the class-order one
    in the eager stage, the counted one always the capacity's; the low-latency split-K follows k"""
    cap = 2048
    stage = _stage(num_out=100)
    lr, ious, feat = _inputs(cap, seed=21)
    g = stage.graphed(cap, C, HW, rle=True, low_latency=low_latency, counted=True)
    g.tar_feat.copy_(feat)
    for k in [2048, 1025, 1024, 1000, 2048]:
        big_lr, big_iou = _poisoned(lr[:k], ious[:k], cap)
        g.lr_masks.copy_(big_lr)
        g.pred_ious.copy_(big_iou)
        out = _replay(g, n=k)
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency)
        _assert_same(out, ref, f"k={k}")
        assert out["counts"]["n_out"] == 100


@pytest.mark.parametrize("low_latency", MODES)
def test_capacity_16384_graph_at_4096(low_latency):
    cap, k = 16384, 4096
    stage = _stage(num_out=100)
    lr, ious, feat = _inputs(k, seed=31)
    g = stage.graphed(cap, C, HW, rle=True, low_latency=low_latency, bind=True, counted=True)
    out = _replay(g, lr_masks=lr, pred_ious=ious, tar_feat=feat)
    ref = _eager(stage, lr, ious, feat, low_latency)
    _assert_same(out, ref, f"k={k}")


@pytest.mark.parametrize("low_latency", MODES)
def test_eager_counted_call_and_its_taps(low_latency):
    """match_async(count_capacity=N) on k-row tensors; the taps keep N rows and get() returns the k live ones, equal to
    the eager stage's, with the fused iou_thr filter"""
    stage = _stage()
    lr, ious, feat = _inputs(200, seed=41)
    for k in (200, 129, 57):
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency, iou_thr=0.5, taps=True)
        out = _eager(stage, lr[:k], ious[:k], feat, low_latency, iou_thr=0.5, taps=True, count_capacity=1100)
        _assert_same(out, ref, f"k={k}")
        for name in ("sim", "obj_feats"):
            assert out["taps"][name].shape == ref["taps"][name].shape, name
            assert torch.equal(out["taps"][name], ref["taps"][name]), name


@pytest.mark.parametrize("low_latency", MODES)
def test_counted_sized_bound_banked_graph(low_latency):
    """one graph: counted (capacity 512), sized, bound and banked (capacity 80, a 7-class bank)"""
    stage = _stage()
    lr, ious, feat = _inputs(512, seed=51)
    gen = torch.Generator().manual_seed(52)
    cen = _centres()
    bank = stage.prepare_bank((cen[torch.arange(7) % cen.shape[0]] + 0.05 * torch.randn(7, C, generator=gen)).unsqueeze(1))
    g = stage.graphed(512, C, (640, 640), iou_thr=0.5, rle=True, low_latency=low_latency, min_hw=(200, 200), bind=True,
                      bank_capacity=(80, 0), counted=True)
    for k, hw in [(512, (480, 640)), (300, (333, 500)), (41, (640, 427)), (300, (200, 200))]:
        big_lr, big_iou = _poisoned(lr[:k], ious[:k], 512)
        out = _replay(g, ori_hw=hw, lr_masks=big_lr[:k], pred_ious=big_iou[:k], tar_feat=feat, bank=bank)
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency, hw=hw, iou_thr=0.5, bank=bank,
                     bank_capacity=(80, 0))
        _assert_same(out, ref, f"k={k} hw={hw}")
        assert int(out["labels"].max()) < 7


def test_replay_checks_the_count_on_the_host():
    stage = _stage()
    lr, ious, feat = _inputs(64, seed=61)
    g = stage.graphed(64, C, HW, bind=True, counted=True)
    with pytest.raises(ValueError):
        g.replay(n=65)
    with pytest.raises(ValueError):
        g.replay(n=-1)
    with pytest.raises(ValueError):
        g.replay(lr_masks=lr[:10], pred_ious=ious[:11])
    with pytest.raises(ValueError):
        g.replay(lr_masks=lr[:10])
    with pytest.raises(ValueError):
        stage.graphed(64, C, HW, n_multi=3, counted=True)
    plain = stage.graphed(64, C, HW)
    with pytest.raises(ValueError):
        plain.replay(n=10)


@pytest.mark.parametrize("bad", [257, -1, 1 << 30])
def test_count_outside_the_capacity_gives_an_empty_result(bad):
    """a value written straight to the device (no bind): empty result, counts[3] = 2, the persistent slots cleared, and
    guard bytes around the inputs and the persistent outputs untouched"""
    cap, num_out = 256, 20
    stage = _stage(num_out=num_out)
    lr, ious, feat = _inputs(cap, seed=71)
    guard = 7
    buf = torch.full((cap + 2, 256, 256), 3.5, dtype=torch.float32, device=DEV)
    buf[1:cap + 1] = lr
    iou_buf = torch.full((cap + 2,), 3.5, dtype=torch.float32, device=DEV)
    iou_buf[1:cap + 1] = ious
    masks = torch.full((num_out + 2, *HW), guard, dtype=torch.uint8, device=DEV)
    masks[1:num_out + 1] = 0
    rect = torch.full((num_out + 2, 4), guard, dtype=torch.int32, device=DEV)
    rect[1:num_out + 1] = 0
    out_bufs = (masks[1:num_out + 1], rect[1:num_out + 1])
    # a first image fills the persistent slots
    first = stage.match_async(buf[1:cap + 1], iou_buf[1:cap + 1], feat, HW, persistent_out=out_bufs, count_capacity=cap)
    assert first.get()["counts"]["n_out"] == num_out
    count = torch.tensor([bad], dtype=torch.int32, device=DEV)
    pend = stage.match_async(buf[1:cap + 1], iou_buf[1:cap + 1], feat, HW, persistent_out=out_bufs, count_capacity=cap,
                             count_dev=count)
    with pytest.raises(RuntimeError, match="candidate count"):
        pend.get()
    assert pend.counts.tolist() == [0, 0, 0, 2]
    assert int(out_bufs[0].count_nonzero()) == 0 and int(out_bufs[1].count_nonzero()) == 0
    for t in (masks, rect):
        assert bool((t[0] == guard).all()) and bool((t[-1] == guard).all())
    for t in (buf, iou_buf):
        assert bool((t[0] == 3.5).all()) and bool((t[-1] == 3.5).all())
    assert torch.equal(buf[1:cap + 1], lr)


def test_count_status_and_size_status_are_both_reported():
    stage = _stage()
    lr, ious, feat = _inputs(64, seed=81)
    hw = torch.tensor([100, 100], dtype=torch.int32, device=DEV)  # below the range
    count = torch.tensor([65], dtype=torch.int32, device=DEV)
    pend = stage.match_async(lr, ious, feat, (480, 640), size_range=(hw, (200, 200)), count_capacity=64, count_dev=count)
    torch.cuda.synchronize()
    assert pend.counts.tolist()[3] == 3
    count.fill_(64)
    pend = stage.match_async(lr, ious, feat, (480, 640), size_range=(hw, (200, 200)), count_capacity=64, count_dev=count)
    torch.cuda.synchronize()
    assert pend.counts.tolist()[3] == 1


@pytest.mark.parametrize("low_latency", MODES)
def test_eager_counted_call_on_an_empty_list(low_latency):
    """the compaction kept nothing: freshly allocated [0, 256, 256] / [0] tensors (no address at all) give an empty
    result and clear the persistent slots an earlier image filled"""
    cap, num_out = 256, 20
    stage = _stage(num_out=num_out)
    lr, ious, feat = _inputs(cap, seed=91)
    out_bufs = (torch.zeros((num_out, *HW), dtype=torch.uint8, device=DEV),
                torch.zeros((num_out, 4), dtype=torch.int32, device=DEV))
    first = stage.match_async(lr, ious, feat, HW, persistent_out=out_bufs, low_latency=low_latency, count_capacity=cap)
    assert first.get()["counts"]["n_out"] == num_out
    empty_lr = torch.empty((0, 256, 256), dtype=torch.float32, device=DEV)
    empty_iou = torch.empty((0,), dtype=torch.float32, device=DEV)
    pend = stage.match_async(empty_lr, empty_iou, feat, HW, persistent_out=out_bufs, rle=True, low_latency=low_latency,
                             count_capacity=cap)
    out = pend.get()
    assert out["counts"] == dict(n_keep=0, n_sel=0, n_out=0)
    assert pend.rle_segmentations() == []
    assert int(out_bufs[0].count_nonzero()) == 0 and int(out_bufs[1].count_nonzero()) == 0


@pytest.mark.parametrize("low_latency", MODES)
def test_counted_graph_with_negative_references(low_latency):
    """negative-reference scoring (80 classes x 3 negatives): both similarity GEMMs and neg_top1 take the live count
    (in low-latency mode each GEMM's split-K follows it), bit for bit against the eager stage at k"""
    cap = 2048
    stage = _stage(num_out=100)
    gen = torch.Generator().manual_seed(93)
    cen = _centres()
    pos = cen[torch.arange(80) % cen.shape[0]] + 0.05 * torch.randn(80, C, generator=gen)
    neg = cen[torch.randint(0, cen.shape[0], (80 * 3,), generator=gen)].reshape(80, 3, C)
    stage.set_prototypes_with_negatives(pos, neg + 0.3 / C ** 0.5 * torch.randn(neg.shape, generator=gen))
    lr, ious, feat = _inputs(cap, seed=94)
    g = stage.graphed(cap, C, HW, rle=True, low_latency=low_latency, bind=True, counted=True)
    for k in [2048, 1025, 1000, 129, 57]:
        big_lr, big_iou = _poisoned(lr[:k], ious[:k], cap)
        out = _replay(g, lr_masks=big_lr[:k], pred_ious=big_iou[:k], tar_feat=feat)
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency)
        _assert_same(out, ref, f"k={k}")
        assert out["counts"]["n_out"] > 0
    for k in (1000, 57):  # the eager counted call, with its taps
        ref = _eager(stage, lr[:k].contiguous(), ious[:k].contiguous(), feat, low_latency, taps=True)
        got = _eager(stage, lr[:k], ious[:k], feat, low_latency, taps=True, count_capacity=cap)
        _assert_same(got, ref, f"eager k={k}")
        for name in ("sim", "obj_feats"):
            assert torch.equal(got["taps"][name], ref["taps"][name]), name
