"""Dense prompt grids: up to 16 384 candidate masks per image (points_per_side 128, NTTT_MAX_CANDIDATES).

NMS keep / sel lists equal the C oracle exactly from 8 193 to 16 384 boxes (the 16 384-box instances of the class-order
sort and the sparse scan); the whole stage at 16 384 agrees with the torch port of the reference on the same GPU in
both launch modes, with the spatial pooling order on and off, and with the fused candidate filter; the fused multimask
selection reads 64 per-batch chunks or one [16 384, 4, 256, 256] buffer (2^32 elements); a bound, sized graph replays
at that size; 16 385 masks are refused before anything is enqueued; and the drop-in model takes the compacting path
when the grid has more decoder batches than the fused path can address.

Memory: the multimask cases hold 17 GB of logits per copy; each test frees its layout before the next one."""
import ctypes
import gc
import importlib
import types

import numpy as np
import pytest
import torch

from golden_util import assert_close_rel, assert_rows_match, assert_same_ranking
from oracle import nttt_oracle as orc
from oracle import ref_torch

DEV = "cuda:0"
N_MAX = 16384


@pytest.fixture(scope="module")
def P():
    return importlib.import_module("no-time-to-train_b200")


@pytest.fixture(scope="module")
def ops(P):
    return importlib.import_module("no-time-to-train_b200.ops")


@pytest.fixture(autouse=True)
def _release():
    yield
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


def _boxes(n, n_cls, seed):
    """Random low-res boxes with planted identical boxes (2, 3), tied scores (2, 3) and a zero-width box (1)."""
    gen = torch.Generator().manual_seed(seed)
    xy = torch.randint(0, 200, (n, 2), generator=gen)
    wh = torch.randint(0, 56, (n, 2), generator=gen)
    box = torch.cat([xy, xy + wh], 1).int()
    box[3] = box[2]
    box[1] = torch.tensor([5, 5, 5, 40])
    scores = torch.rand(n, generator=gen)
    scores[3] = scores[2]
    labels = torch.randint(0, n_cls, (n,), generator=gen).int()
    top = torch.rand(n, generator=gen) - 0.2
    return box, scores, labels, top


def _equal_up_to_score_ties(want, tv, scores, planted=()):
    if np.array_equal(want, tv):
        return
    assert len(want) == len(tv)
    assert np.array_equal(scores[want], scores[tv]), "kept scores differ from torchvision beyond tie order"
    diff = set(want.tolist()) ^ set(tv.tolist())
    assert diff <= set(planted), diff


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("n_cls", [80, 5, 1])
def test_oracle_box_nms_matches_torchvision_at_16384(n_cls):
    from torchvision.ops import batched_nms
    box, scores, labels, _ = _boxes(N_MAX, n_cls, seed=16384 + n_cls)
    want = orc.box_nms(box.float().numpy(), scores.numpy(), labels.long().numpy(), 0.5)
    tv = batched_nms(box.float(), scores, labels.long(), 0.5).numpy()
    assert 0 < len(want) < N_MAX
    _equal_up_to_score_ties(want, tv, scores.numpy(), planted={2, 3})


# ------------------------------------------------------------------------------------------------ NMS per op
def _nms_against_oracle(ops, box, scores, labels, top, max_keep):
    keep, sel, counts = ops.box_nms(box.to(DEV), scores.to(DEV), labels.to(DEV), top.to(DEV), 0.5, max_keep)
    nk, ns = counts.cpu().tolist()
    want = orc.box_nms(box.float().numpy(), scores.numpy(), labels.long().numpy(), 0.5)[:max_keep]
    assert nk == len(want) and np.array_equal(keep.cpu().numpy()[:nk], want)
    want_sel = want[top.numpy()[want] > 0]
    assert ns == len(want_sel) and np.array_equal(sel.cpu().numpy()[:ns], want_sel)
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("max_keep", [800, None])
@pytest.mark.parametrize("n_cls", [80, 5, 1])
@pytest.mark.parametrize("n", [8193, 12000, 16384])
def test_box_nms_long_lists_match_oracle(ops, n, n_cls, max_keep):
    box, scores, labels, top = _boxes(n, n_cls, seed=n * 7 + n_cls)
    _nms_against_oracle(ops, box, scores, labels, top, max_keep or n)


@pytest.mark.gpu
@pytest.mark.parametrize("max_keep", [800, N_MAX])
def test_box_nms_one_class_chain_as_long_as_the_list(ops, max_keep):
    """The scan's worst case: one class, boxes along a line, each overlapping only its neighbours (IoU 7/13), so
    keep / suppress alternates along a dependency chain through all 512 chunks."""
    n = N_MAX
    x0 = torch.arange(n) * 3
    box = torch.stack([x0, torch.zeros(n, dtype=torch.long), x0 + 10, torch.full((n,), 10)], 1).int()
    scores = torch.linspace(1.0, 0.01, n)
    labels = torch.zeros(n, dtype=torch.int32)
    top = torch.rand(n, generator=torch.Generator().manual_seed(3)) - 0.3
    want = _nms_against_oracle(ops, box, scores, labels, top, max_keep)
    assert want[:3].tolist() == [0, 2, 4] and len(want) == min(max_keep, n // 2)


# ------------------------------------------------------------------------------------------------ refusal
@pytest.mark.gpu
def test_more_than_16384_candidates_are_refused_before_any_launch(P):
    lib = P._lib.load()
    n = N_MAX + 1
    assert P._lib.MAX_CANDIDATES == N_MAX
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=10, enc_hw=(37, 37)))
    stage.set_prototypes(torch.randn(3, 1, 64))
    dummy = torch.zeros((1 << 20,), dtype=torch.uint8, device=DEV)  # addresses that must never be read
    sentinel = torch.full((4,), -7, dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    launches = lib.nttt_launch_count()
    stream = torch.cuda.current_stream().cuda_stream
    p = dummy.data_ptr()
    # nttt_box_nms
    assert lib.nttt_box_nms(p, p, p, p, n, 0.5, 100, p, sentinel.data_ptr(), p, sentinel.data_ptr() + 4, p,
                            dummy.numel(), stream) == -5  # NTTT_EUNSUPPORTED
    # the three whole-image entries
    a = P._lib.MatchArgs()
    a.logits, a.pred_ious, a.tar_feat, a.proto = p, p, p, p
    a.n, a.lr_h, a.lr_w, a.eh, a.ew, a.c, a.n_cls = n, 256, 256, 37, 37, 64, 3
    a.ori_h, a.ori_w, a.nms_thr, a.num_out_instance, a.max_sel = 480, 640, 0.5, 10, 80
    a.out_masks, a.out_boxes, a.out_scores, a.out_labels, a.out_index = p, p, p, p, p
    a.counts, a.workspace, a.workspace_bytes = sentinel.data_ptr(), p, dummy.numel()
    assert lib.nttt_match_image(stage.ctx, ctypes.byref(a), stream) == -5
    rng = P._lib.MatchSizeRange(p, 100, 100)
    assert lib.nttt_match_image_sized(stage.ctx, ctypes.byref(a), ctypes.byref(rng), stream) == -5
    assert lib.nttt_match_image_bound(stage.ctx, ctypes.byref(a), None, p, stream) == -5
    torch.cuda.synchronize()
    assert lib.nttt_launch_count() == launches
    assert sentinel.cpu().tolist() == [-7] * 4
    # the Python API, before it allocates or enqueues anything
    lr = torch.empty((n, 256, 256), device=DEV)
    with pytest.raises(ValueError, match="16384"):
        stage.match_async(lr, torch.empty((n,), device=DEV), torch.empty((37 * 37, 64), device=DEV), (480, 640))
    with pytest.raises(ValueError, match="16384"):
        stage.match_async([torch.empty((n, 2, 8, 8), device=DEV)], None, torch.empty((37 * 37, 64), device=DEV), (480, 640),
                          multi_ious=torch.empty((n, 2), device=DEV))
    with pytest.raises(ValueError, match="16384"):
        stage.graphed(n, 64, (480, 640))
    torch.cuda.synchronize()
    assert lib.nttt_launch_count() == launches


# ------------------------------------------------------------------------------------------------ whole stage
@pytest.fixture(scope="module")
def dense_inputs(synth):
    """16 384 candidates at config-2 shapes (ViT-L width, 80 classes, 1024 x 1024), clustered, with the degenerate
    masks of synth.inject_degenerate_cases."""
    return synth.make_stage_inputs(N_MAX, 1024, 80, 10, (1024, 1024), seed=1616, clustered=True, degenerate=True)


def _dense_stage(P, inp, num_out=100):
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=num_out, enc_hw=(37, 37)))
    stage.set_prototypes(inp.feats_ins_avg)
    return stage


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["low_latency", "throughput_ordered", "throughput_unordered"])
def test_stage_at_16384_against_torch_port_on_gpu(P, dense_inputs, mode):
    """As test_full_size_against_torch_port_on_gpu, at 16 384 masks: similarities within the tolerance, then
    everything downstream (NMS keep and selection counts, ranking, masks, boxes) conditioned on the same similarities."""
    inp = dense_inputs
    stage = _dense_stage(P, inp)
    if mode != "low_latency":
        stage.tune("pool_order", 1 if mode == "throughput_ordered" else 0)
    lr, ious, feat = inp.lr_masks.to(DEV), inp.pred_ious.to(DEV), inp.tar_feat.to(DEV)
    out = stage.match(lr, ious, feat, inp.ori_hw, taps=True, low_latency=mode == "low_latency")
    cfg = ref_torch.StageConfig(num_out_instance=100)
    with torch.inference_mode():
        free = ref_torch.match_image(lr, ious, feat, inp.feats_ins_avg.to(DEV), cfg, inp.ori_hw)
    sim_ref, sim_got = free["aux"]["sim"].cpu().numpy(), out["taps"]["sim"].cpu().numpy()
    assert_close_rel(sim_got, sim_ref, what="sim")
    assert_close_rel(out["taps"]["obj_feats"].cpu().numpy(), free["aux"]["obj_feats"].cpu().numpy(), what="obj_feats")
    lab_ref, lab_got = sim_ref.argmax(1), sim_got.argmax(1)
    for i in np.nonzero(lab_ref != lab_got)[0]:
        assert abs(sim_ref[i, lab_ref[i]] - sim_ref[i, lab_got[i]]) <= 1e-5, "label flip outside a float near-tie"
    del free
    with torch.inference_mode():
        ref = ref_torch.match_image(lr, ious, feat, inp.feats_ins_avg.to(DEV), cfg, inp.ori_hw,
                                    override=dict(sim=out["taps"]["sim"], obj_feats=out["taps"]["obj_feats"]))
    assert out["counts"]["n_keep"] == ref["aux"]["keep"].numel()
    assert out["counts"]["n_sel"] == ref["aux"]["sel_index"].numel()
    assert_same_ranking(out["scores"].cpu().numpy(), out["labels"].cpu().numpy(), ref["scores"].cpu().numpy(),
                        ref["labels"].cpu().numpy(), what=mode)
    m = out["binary_masks"]
    assert m.shape[0] > 0
    assert torch.equal(m, ref_torch.upsample_threshold(lr[out["index"].long()], inp.ori_hw))
    assert torch.equal(out["bboxes"], ref_torch.mask_boxes(m))


@pytest.mark.gpu
def test_fused_filter_at_16384_drops_most_candidates(P, dense_inputs):
    """The iou gate with ~90 % of the candidates filtered out: the filtered boxes carry the unique labels -2 - i down to
    -2 - 16383 in the class-order NMS; the result is the reference's compaction followed by the stage."""
    inp = dense_inputs
    thr = 0.9
    gen = torch.Generator().manual_seed(17)
    ious = torch.rand(N_MAX, generator=gen)
    keep = ious > thr
    assert 1000 < int(keep.sum()) < 2500
    stage = _dense_stage(P, inp)
    lr, feat = inp.lr_masks.to(DEV), inp.tar_feat.to(DEV)
    got = stage.match(lr, ious.to(DEV), feat, inp.ori_hw, iou_thr=thr, taps=True, low_latency=False)
    kept = torch.nonzero(keep).flatten().to(DEV)
    with torch.inference_mode():
        ref = ref_torch.match_image(lr[kept], ious.to(DEV)[kept], feat, inp.feats_ins_avg.to(DEV),
                                    ref_torch.StageConfig(num_out_instance=100), inp.ori_hw,
                                    override=dict(sim=got["taps"]["sim"][kept], obj_feats=got["taps"]["obj_feats"][kept]))
    assert got["counts"]["n_keep"] == ref["aux"]["keep"].numel()
    assert got["counts"]["n_sel"] == ref["aux"]["sel_index"].numel()
    assert_same_ranking(got["scores"].cpu().numpy(), got["labels"].cpu().numpy(), ref["scores"].cpu().numpy(),
                        ref["labels"].cpu().numpy(), what="filtered")
    orig_index = kept[ref["aux"]["sel_index"][ref["aux"]["order"]]]
    assert_rows_match(dict(scores=got["scores"], labels=got["labels"], bboxes=got["bboxes"], masks=got["binary_masks"],
                           index=got["index"]),
                      dict(scores=ref["scores"], labels=ref["labels"], bboxes=ref["bboxes"], masks=ref["binary_masks"],
                           index=orig_index), what="filtered")


# ------------------------------------------------------------------------------------------------ fused multimask
M, CHUNK = 4, 256


def _decoder_chunks(synth, n, seed, centres):
    """The decoder's raw output for n prompts, generated on the device chunk by chunk: separate [256, 4, 256, 256]
    allocations (m jittered variants of one blob per prompt, as synth.make_multimask_inputs) and ious [n, 4]."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    chunks = []
    for k in range(n // CHUNK):
        base, _, _ = synth.make_stage_inputs_device(CHUNK, centres, DEV, seed=seed * 1000 + k)
        ch = torch.empty((CHUNK, M, 256, 256), dtype=torch.float32, device=DEV)
        for j in range(M):
            ch[:, j] = base * (1.0 + 0.1 * j) + 0.35 * (j + 1) * torch.randn((CHUNK, 1, 1), generator=gen, device=DEV)
        chunks.append(ch)
    ious = 0.2 + 0.8 * torch.rand((n, M), generator=gen, device=DEV)
    return chunks, ious


def _same(out, ref, what):
    assert out["counts"] == ref["counts"], what
    assert torch.equal(torch.isnan(out["scores"]), torch.isnan(ref["scores"])), what
    assert torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(ref["scores"])), what
    for key in ("labels", "bboxes", "index", "binary_masks"):
        assert torch.equal(out[key], ref[key]), (what, key)


@pytest.mark.gpu
def test_fused_multimask_at_16384_prompts_in_both_layouts(P, synth):
    """64 chunks of [256, 4, 256, 256], then one [16 384, 4, 256, 256] buffer (2^32 elements, plane offsets past 2^32
    bytes): both equal the single-plane call on the planes torch's argmax picks, filter included."""
    centres = synth.cluster_centres(1024)
    feat = synth.make_stage_inputs_device(8, centres, DEV, seed=5)[2]
    protos = (centres[torch.arange(80) % centres.shape[0]] + 0.05 * torch.randn(80, 1024, generator=torch.Generator()
                                                                               .manual_seed(6))).unsqueeze(1)
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=100, enc_hw=(37, 37)))
    stage.set_prototypes(protos)
    hw, thr = (1024, 1024), 0.5
    chunks, ious = _decoder_chunks(synth, N_MAX, 7, centres)
    assert len(chunks) == P._lib.MAX_CHUNKS
    best = torch.argmax(ious[:, 1:], dim=-1) + 1
    planes = torch.empty((N_MAX, 256, 256), dtype=torch.float32, device=DEV)
    for k, ch in enumerate(chunks):
        rows = slice(k * CHUNK, (k + 1) * CHUNK)
        planes[rows] = ch[torch.arange(CHUNK, device=DEV), best[rows]]
    score = ious[torch.arange(N_MAX, device=DEV), best].contiguous()
    want = stage.match(planes, score, feat, hw, iou_thr=thr)
    del planes
    assert want["counts"]["n_out"] == 100
    got = stage.match(chunks, None, feat, hw, iou_thr=thr, multi_ious=ious, multi_first=1)
    _same(got, want, "64 chunks")
    # one buffer: the same values (each chunk released once copied)
    one = torch.empty((N_MAX, M, 256, 256), dtype=torch.float32, device=DEV)
    assert one.numel() == 1 << 32
    for k in range(len(chunks)):
        one[k * CHUNK:(k + 1) * CHUNK] = chunks[k]
        chunks[k] = None
    del chunks
    got = stage.match(one, None, feat, hw, iou_thr=thr, multi_ious=ious, multi_first=1)
    _same(got, want, "one buffer")


@pytest.mark.gpu
def test_bound_sized_graph_at_16384_with_64_chunks(P, synth):
    centres = synth.cluster_centres(1024)
    protos = (centres[torch.arange(80) % centres.shape[0]] + 0.05 * torch.randn(80, 1024, generator=torch.Generator()
                                                                               .manual_seed(8))).unsqueeze(1)
    stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=100, enc_hw=(37, 37)))
    stage.set_prototypes(protos)
    cap = (1024, 1024)
    g = stage.graphed(N_MAX, 1024, cap, iou_thr=0.5, n_multi=M, min_hw=(200, 200), bind=True,
                      chunk_prompts=CHUNK).capture()
    assert len(g.lr_masks) == 64
    # input set 1: the producer's own chunks, bound at replay; input set 2: written into the graph's static buffers
    chunks, ious = _decoder_chunks(synth, N_MAX, 9, centres)
    feat = synth.make_stage_inputs_device(8, centres, DEV, seed=10)[2]
    hw = (768, 1024)
    out = g.replay(ori_hw=hw, lr_masks=chunks, multi_ious=ious, tar_feat=feat).get()
    eager = stage.match(chunks, None, feat, hw, iou_thr=0.5, multi_ious=ious, multi_first=1, low_latency=False)
    assert eager["counts"]["n_out"] > 0
    _same(out, eager, "bound chunks")
    want = torch.zeros_like(g._out[0].view(torch.bool))
    k, h, w = eager["binary_masks"].shape
    want[:k, :h, :w] = eager["binary_masks"]
    assert torch.equal(g._out[0].view(torch.bool), want)
    del chunks, eager
    chunks2, ious2 = _decoder_chunks(synth, N_MAX, 11, centres)
    for dst, src in zip(g.lr_masks, chunks2):
        dst.copy_(src)
    del chunks2
    g.multi_ious.copy_(ious2)
    g.tar_feat.copy_(synth.make_stage_inputs_device(8, centres, DEV, seed=12)[2])
    hw = (1024, 640)
    out = g.replay(ori_hw=hw).get()
    eager = stage.match(g.lr_masks, None, g.tar_feat, hw, iou_thr=0.5, multi_ious=g.multi_ious, multi_first=1,
                        low_latency=False)
    assert eager["counts"]["n_out"] > 0
    _same(out, eager, "static buffers")


# ------------------------------------------------------------------------------------------------ drop-in class
@pytest.mark.gpu
def test_model_takes_the_compacting_path_beyond_64_decoder_batches(P, synth):
    """points_per_side 128: testing_point_bs 256 gives 64 decoder batches (the fused path), 128 gives 128 batches (the
    compacting `_forward_sam` path).  Every prompt passes the iou gate here, so both hand the stage the same 16 384
    candidates and the result dicts are identical."""
    centres = synth.cluster_centres(1024)
    chunks, ious = _decoder_chunks(synth, N_MAX, 13, centres)
    multi = torch.cat(chunks)
    del chunks
    ious = ious * 0.5 + 0.45  # all above the iou_thr 0.4 below
    feat = synth.make_stage_inputs_device(8, centres, DEV, seed=14)[2]
    n_cls = 80
    protos = (centres[torch.arange(n_cls) % centres.shape[0]] + 0.05 * torch.randn(n_cls, 1024, generator=torch.Generator()
                                                                                   .manual_seed(15))).unsqueeze(1)

    def run(bs):
        calls = {"i": 0}

        def decoder(**kw):
            i = calls["i"]
            calls["i"] += 1
            return multi[i * bs:(i + 1) * bs].clone(), ious[i * bs:(i + 1) * bs].clone(), None, None

        prompt_encoder = lambda points, boxes, masks: (torch.zeros(bs, 2, 4, device=DEV),
                                                       torch.zeros(bs, 4, 2, 2, device=DEV))
        prompt_encoder.get_dense_pe = lambda: torch.zeros(1, 4, 2, 2, device=DEV)
        pred = types.SimpleNamespace(
            forward_image=lambda imgs: {},
            _prepare_backbone_features=lambda bo: (None, [torch.zeros(16, 1, 4, device=DEV),
                                                          torch.zeros(4, 1, 4, device=DEV)], None, [(4, 4), (2, 2)]),
            sam_prompt_encoder=prompt_encoder, sam_mask_decoder=decoder)

        class Model(P.Sam2MatchingBaselineNoAMG):
            def _extract_target_features(self, tar_img, device):
                return feat, tar_img.to(device)

        m = Model(sam2_infer_cfgs=dict(points_per_side=128, testing_point_bs=bs, iou_thr=0.4, nms_thr=0.5,
                                       num_out_instance=100, kmeans_k=2, n_pca_components=2, cls_num_per_mask=1),
                  memory_bank_cfg=dict(enable=True, category_num=n_cls, length=1),
                  encoder_geometry=(518, 14, 1024), predictor=pred, device=DEV)
        m.output_ring = 0
        m.memory_bank.feats_ins_avg.copy_(protos)
        m.memory_bank.postprocessed[0] = True
        info = dict(ori_height=1024, ori_width=1024, file_name="x", id=0)
        out = m([dict(data_mode="test", target_img=torch.zeros(3, 64, 64), target_img_info=info)])[0]
        assert calls["i"] == N_MAX // bs
        return out

    fused, compacted = run(256), run(128)
    assert fused["binary_masks"].shape[0] == 100
    for key in ("binary_masks", "bboxes", "labels"):
        assert torch.equal(fused[key], compacted[key]), key
    assert torch.equal(torch.nan_to_num(fused["scores"]), torch.nan_to_num(compacted["scores"]))
    assert torch.equal(torch.isnan(fused["scores"]), torch.isnan(compacted["scores"]))
