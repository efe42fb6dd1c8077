"""A captured stage with its memory bank bound at replay (`MatchingStage.graphed(..., bank_capacity=...)`,
`nttt_match_bank_bind`, `nttt_match_image_banked`): one capture scores images against banks of any class count up to
the capacity.  Every replay gives bit for bit what the eager banked stage gives on the same bank and inputs; a bank at
the capacity gives what the unbanked stage gives; a bank below it stays within the similarity bound of the float64
reference, and its padded columns never win.  Malformed banks are rejected on the host before anything is enqueued."""
import importlib

import pytest
import torch

from gemm_ref import TOL_SIM, check_labels, normalised_error
from golden_util import assert_rows_match
from oracle import ref_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CAP = 80  # class capacity of the graphs (config-2: COCO's 80 classes)
N, C = 128, 384
HW = (480, 640)
MODES = [False, True]  # low_latency


def _pkg():
    return importlib.import_module("no-time-to-train_b200")


def _inputs(seed, n=N, c=C, n_cls=CAP):
    P = _pkg()
    inp = P.synth.make_stage_inputs(n, c, n_cls, 2, (1, 1), seed=seed, clustered=True, degenerate=2)
    gen = torch.Generator().manual_seed(seed + 1)
    inp.pred_ious = torch.rand(n, generator=gen) * 0.6 + 0.4  # about a sixth fall below the 0.5 threshold
    inp.pred_ious[8:15] = 0.99  # the border cases reach the output
    return inp


def _dev(inp):
    return inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV)


def _stage(num_out=20):
    P = _pkg()
    return P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=num_out, enc_hw=(37, 37)))


def _feats(inp, k, seed):
    """feats_ins_avg of a k-class bank: k of the input's 80 classes in a seeded order, with small per-shot noise (one
    bank of a seed sweep)"""
    gen = torch.Generator().manual_seed(seed)
    pick = torch.randperm(inp.feats_ins_avg.shape[0], generator=gen)[:k]
    return inp.feats_ins_avg[pick] + (0.02 / C ** 0.5) * torch.randn(k, *inp.feats_ins_avg.shape[1:], generator=gen)


def _neg_feats(inp, k, l_neg, seed):
    """(feats_avg [k, c], feats_ins_avg_neg [k, l_neg, c]) of a negative-reference bank"""
    gen = torch.Generator().manual_seed(seed)
    perm = torch.randperm(inp.feats_ins_avg.shape[0], generator=gen)
    pos = inp.feats_ins_avg[perm[:k]].mean(1)
    neg = inp.feats_ins_avg[perm[torch.randint(0, perm.numel(), (k * l_neg,), generator=gen)], 0].reshape(k, l_neg, -1)
    return pos, neg + (0.3 / C ** 0.5) * torch.randn(neg.shape, generator=gen)


def _eager(stage, inputs, bank, cap, low_latency, hw=HW, taps=False, **kw):
    """the eager banked call (`match_async(bank=..., bank_capacity=...)`), with its RLE"""
    lr, ious, feat = inputs
    pend = stage.match_async(lr, ious, feat, hw, iou_thr=0.5, rle=True, taps=taps, low_latency=low_latency, bank=bank,
                             bank_capacity=cap, **kw)
    out = pend.get()
    out["segmentations"] = pend.rle_segmentations()
    return out


def _replay(g, **kw):
    pend = g.replay(**kw)
    out = pend.get()
    out["segmentations"] = pend.rle_segmentations()
    return out


def _unbanked(stage, inputs, low_latency, feats=None, neg=None):
    """today's path: the unbanked entry after set_prototypes*"""
    if neg is None:
        stage.set_prototypes(feats)
    else:
        stage.set_prototypes_with_negatives(*neg)
    return stage.match(*inputs, HW, iou_thr=0.5, rle=True, low_latency=low_latency)


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


def _identical(out, ref) -> bool:
    try:
        _assert_same(out, ref, "")
        return True
    except AssertionError:
        return False


def _rows(out):
    return dict(scores=out["scores"], labels=out["labels"], bboxes=out["bboxes"], masks=out["binary_masks"],
                index=out["index"])


@pytest.mark.parametrize("low_latency", MODES)
def test_one_banked_graph_serves_many_banks(low_latency):
    inp = _inputs(101)
    stage = _stage()
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bank_capacity=(CAP, 0))
    g.lr_masks.copy_(inputs[0])
    g.pred_ious.copy_(inputs[1])
    g.tar_feat.copy_(inputs[2])
    graph = None
    for step, k in enumerate([7, 1, 40, 80, 7, 2, 80]):
        bank = stage.prepare_bank(_feats(inp, k, 110 + step))
        out = _replay(g, bank=bank)
        if graph is None:
            graph = g.graph
        assert g.graph is graph  # (one capture serves every bank)
        assert g.pending._bank is bank  # held until the next replay
        ref = _eager(stage, inputs, bank, (CAP, 0), low_latency)
        _assert_same(out, ref, f"bank {step} ({k} classes)")
        assert out["counts"]["n_out"] > 0
        assert int(out["labels"].max()) < k


@pytest.mark.parametrize("low_latency", MODES)
def test_one_negative_reference_graph_serves_many_banks(low_latency):
    inp = _inputs(151)
    stage = _stage()
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bank_capacity=(CAP, 3))
    g.lr_masks.copy_(inputs[0])
    g.pred_ious.copy_(inputs[1])
    g.tar_feat.copy_(inputs[2])
    for step, (k, l_neg) in enumerate([(7, 2), (1, 1), (40, 3), (80, 3), (80, 1)]):
        bank = stage.prepare_bank_with_negatives(*_neg_feats(inp, k, l_neg, 160 + step))
        out = _replay(g, bank=bank)
        ref = _eager(stage, inputs, bank, (CAP, 3), low_latency)
        _assert_same(out, ref, f"negative bank {step} ({k} x {l_neg})")
        assert out["counts"]["n_out"] > 0


@pytest.mark.parametrize("low_latency", MODES)
def test_bank_at_capacity_equals_the_unbanked_entry(low_latency):
    """live counts equal to the capacity: the launch shapes are those of the unbanked entry, so are the results"""
    inp = _inputs(201)
    stage = _stage()
    inputs = _dev(inp)
    feats = _feats(inp, CAP, 202)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True, bank_capacity=(CAP, 0))
    out = _replay(g, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2], bank=stage.prepare_bank(feats))
    _assert_same(out, _unbanked(stage, inputs, low_latency, feats=feats), "plain")
    neg = _neg_feats(inp, CAP, 3, 203)
    gn = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True, bank_capacity=(CAP, 3))
    out = _replay(gn, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2],
                  bank=stage.prepare_bank_with_negatives(*neg))
    _assert_same(out, _unbanked(stage, inputs, low_latency, neg=neg), "negative references")
    assert out["counts"]["n_out"] > 0


@pytest.mark.parametrize("low_latency", MODES)
def test_bank_below_capacity_against_float64_and_the_unbanked_entry(low_latency):
    inp = _inputs(301)
    stage = _stage()
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True, bank_capacity=(CAP, 0))
    for k in (7, 40):
        feats = _feats(inp, k, 310 + k)
        bank = stage.prepare_bank(feats)
        # the live similarities against the float64 product of the obj_feats tap with the float64 prototypes
        pend = stage.match_async(*inputs, HW, iou_thr=0.5, taps=True, low_latency=low_latency, bank=bank,
                                 bank_capacity=(CAP, 0))
        assert pend.taps["sim"].shape == (N, CAP)
        taps = pend.get()["taps"]
        sim, obj = taps["sim"], taps["obj_feats"]
        assert sim.shape == (N, k)
        o64, p64 = obj.double(), ref_torch.prototypes(feats.double()).to(DEV)
        ref, bound = o64 @ p64.t(), o64.abs() @ p64.abs().t()
        assert normalised_error(sim, ref, bound, f"sim, {k} of {CAP}") <= TOL_SIM
        check_labels(sim, ref, bound, f"sim, {k} of {CAP}")
        # the graph's outputs against today's path on the same bank
        out = _replay(g, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2], bank=bank)
        ref_out = _unbanked(stage, inputs, low_latency, feats=feats)
        assert out["counts"] == ref_out["counts"]
        assert out["counts"]["n_out"] > 0
        assert_rows_match(_rows(out), _rows(ref_out), what=f"{k} of {CAP} classes vs unbanked")
        print(f"[bank below capacity] {k} of {CAP} classes, low_latency={low_latency}: bit-identical to the unbanked "
              f"entry: {_identical(out, ref_out)}")


@pytest.mark.parametrize("low_latency", MODES)
def test_padded_columns_never_win(low_latency):
    """Prototypes anti-aligned with every pooled feature: every live similarity is negative, so a padded column
    (similarity 0) would beat them all.  No score passes the `> 0` filter, so the labels show in class-aware NMS: the
    keep count must be the unbanked entry's, and a bank whose extra class is a zero row (what a padded column winning
    would give: every mask in one class) must keep fewer masks."""
    inp = _inputs(401)
    gen = torch.Generator().manual_seed(402)
    k, width = 7, C // 7
    # positive features: patches in vertical stripes of 3 encoder columns, stripe s weighted on channel block s % k; every
    # pooled row has positive entries, and its heaviest block follows where the mask lies
    block = (torch.arange(37).repeat(37) // 3) % k
    tar = 0.05 + 0.01 * torch.rand(37 * 37, C, generator=gen)
    for b in range(k):
        tar[block == b, b * width:(b + 1) * width] += 1.0
    inp.tar_feat = tar
    # negative prototypes, lightest on their own block: class j scores least negative on masks heaviest on block j
    feats = -(1.0 + 0.01 * torch.rand(k, 2, C, generator=gen))
    for j in range(k):
        feats[j, :, j * width:(j + 1) * width] = -0.05
    stage = _stage()
    inputs = _dev(inp)
    bank = stage.prepare_bank(feats)
    pend = stage.match_async(*inputs, HW, iou_thr=0.5, taps=True, low_latency=low_latency, bank=bank,
                             bank_capacity=(CAP, 0))
    sim = pend.get()["taps"]["sim"]
    nonempty = sim.abs().amax(1) > 0
    assert nonempty.sum() > N // 2 and bool((sim[nonempty] < 0).all())
    labels = sim.argmax(1)
    assert labels[nonempty].unique().numel() > 1  # (the live labels are not all one class)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bank_capacity=(CAP, 0))
    g.lr_masks.copy_(inputs[0])
    g.pred_ious.copy_(inputs[1])
    g.tar_feat.copy_(inputs[2])
    out = _replay(g, bank=bank)
    _assert_same(out, _eager(stage, inputs, bank, (CAP, 0), low_latency), "eager banked")
    ref = _unbanked(stage, inputs, low_latency, feats=feats)
    _assert_same(out, ref, "unbanked")
    assert out["counts"]["n_sel"] == 0
    padded_wins = _unbanked(stage, inputs, low_latency, feats=torch.cat([feats, torch.zeros(1, 2, C)]))
    assert padded_wins["counts"]["n_keep"] < out["counts"]["n_keep"]


@pytest.mark.parametrize("low_latency", MODES)
def test_one_and_two_class_banks_in_a_wide_graph(low_latency):
    """The `k == n_cls` rule follows the live class count.  (It only rescales scores <= 0, which the `> 0` filter
    drops, so what shows is that one- and two-class banks give what the unbanked entry gives.)"""
    inp = _inputs(501)
    stage = _stage()
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True, bank_capacity=(CAP, 0))
    for k in (1, 2):
        feats = _feats(inp, k, 510 + k)
        out = _replay(g, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2], bank=stage.prepare_bank(feats))
        ref = _unbanked(stage, inputs, low_latency, feats=feats)
        assert out["counts"] == ref["counts"] and out["counts"]["n_out"] > 0
        assert_rows_match(_rows(out), _rows(ref), what=f"{k} class(es) of {CAP}")
        assert int(out["labels"].max()) < k
        print(f"[small bank] {k} of {CAP} classes, low_latency={low_latency}: bit-identical to the unbanked entry: "
              f"{_identical(out, ref)}")


@pytest.mark.parametrize("low_latency", MODES)
def test_banked_bound_sized_graph(low_latency):
    """banked + bound (the decoder's chunk list) + sized: sizes, input sets and banks all change between replays"""
    P = _pkg()
    n, m, cp = 64, 4, 24
    inp = _inputs(601, n=n)
    stage = _stage()
    g = stage.graphed(n, C, (1024, 1024), iou_thr=0.5, rle=True, n_multi=m, low_latency=low_latency, min_hw=(176, 160),
                      bind=True, chunk_prompts=cp, bank_capacity=(CAP, 0))
    for step, (hw, k) in enumerate([((1024, 1024), 80), ((200, 180), 7), ((480, 640), 40), ((1024, 300), 1),
                                    ((333, 500), 7)]):
        multi, ious = P.synth.make_multimask_inputs(n, m, seed=610 + step)
        chunks = [t.to(DEV) for t in multi.split(cp)]
        gen = torch.Generator().manual_seed(620 + step)
        feat = (inp.tar_feat + (0.3 / C ** 0.5) * torch.randn(inp.tar_feat.shape, generator=gen)).to(DEV)
        ious = ious.to(DEV)
        bank = stage.prepare_bank(_feats(inp, k, 630 + step))
        out = _replay(g, ori_hw=hw, lr_masks=chunks, multi_ious=ious, tar_feat=feat, bank=bank)
        ref = _eager(stage, (chunks, None, feat), bank, (CAP, 0), low_latency, hw=hw, multi_ious=ious, multi_first=1)
        _assert_same(out, ref, (hw, k))
        assert out["counts"]["n_out"] > 0


@pytest.mark.parametrize("low_latency", MODES)
def test_set_prototypes_does_not_recapture_a_banked_graph(low_latency):
    inp = _inputs(701)
    stage = _stage()
    stage.set_prototypes(_feats(inp, 9, 702))
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, low_latency=low_latency, bind=True, bank_capacity=(CAP, 0))
    out = _replay(g, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2])
    graph = g.graph
    _assert_same(out, _eager(stage, inputs, None, (CAP, 0), low_latency), "first prototypes")
    first = out["labels"].clone()
    for step in range(2):
        stage.set_prototypes(_feats(inp, 9 + 20 * step, 710 + step))
        out = _replay(g, lr_masks=inputs[0], pred_ious=inputs[1], tar_feat=inputs[2])  # (no bank: the stage's)
        assert g.graph is graph
        _assert_same(out, _eager(stage, inputs, None, (CAP, 0), low_latency), f"replaced prototypes {step}")
        if step == 0:
            assert not torch.equal(out["labels"], first)  # (the bank decides the result)


def test_malformed_banks_raise_before_enqueueing():
    inp = _inputs(801)
    stage = _stage()
    inputs = _dev(inp)
    g = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, bank_capacity=(CAP, 0))
    gn = stage.graphed(N, C, HW, iou_thr=0.5, rle=True, bank_capacity=(CAP, 2))
    for graph in (g, gn):
        graph.lr_masks.copy_(inputs[0])
        graph.pred_ious.copy_(inputs[1])
        graph.tar_feat.copy_(inputs[2])
    P = _pkg()
    PreparedBank = P.matching.PreparedBank
    bank = stage.prepare_bank(_feats(inp, 7, 802))
    nbank = stage.prepare_bank_with_negatives(*_neg_feats(inp, 7, 2, 803))
    assert _replay(g, bank=bank)["counts"]["n_out"] > 0
    assert _replay(gn, bank=nbank)["counts"]["n_out"] > 0
    structs = (g.bank_dev.clone(), gn.bank_dev.clone())
    p = bank.proto
    bad = [
        (g, stage.prepare_bank(torch.randn(7, 2, 256))),                           # channels
        (g, PreparedBank(p.cpu(), None, 7, 0, C)),                                 # device
        (g, PreparedBank(p.double(), None, 7, 0, C)),                              # dtype
        (g, PreparedBank(p.t().contiguous().t(), None, 7, 0, C)),                  # not contiguous
        (g, PreparedBank(p[:5], None, 7, 0, C)),                                   # shape
        (g, stage.prepare_bank(_feats(inp, CAP, 804).repeat(2, 1, 1)[:CAP + 1])),  # n_cls above the capacity
        (g, nbank),                                                                # negatives in a plain graph
        (gn, bank),                                                                # a plain bank in a negative graph
        (gn, stage.prepare_bank_with_negatives(*_neg_feats(inp, 7, 3, 805))),      # l_neg above the capacity
        (g, "not a bank"),
    ]
    for graph, b in bad:
        with pytest.raises((TypeError, ValueError)):
            graph.replay(bank=b)
    unbanked = stage.graphed(N, C, HW, iou_thr=0.5)
    with pytest.raises(ValueError, match="bank_capacity"):
        unbanked.replay(bank=bank)
    assert unbanked.graph is None  # (nothing captured)
    with pytest.raises(ValueError):
        stage.match_async(*inputs, HW, bank=bank)  # a bank needs the banked entry
    with pytest.raises(ValueError):
        stage.match_async(*inputs, HW, bank=nbank, bank_capacity=(CAP, 0))
    torch.cuda.synchronize()
    assert torch.equal(g.bank_dev, structs[0]) and torch.equal(gn.bank_dev, structs[1])  # nothing was bound
    for graph, b, cap in ((g, bank, (CAP, 0)), (gn, nbank, (CAP, 2))):
        _assert_same(_replay(graph, bank=b), _eager(stage, inputs, b, cap, False), "after the rejections")
