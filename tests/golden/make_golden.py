"""Generate golden vectors by executing the REAL reference code on seeded synthetic inputs.

Run in the authoring container only (needs /root/reference):

    python tests/golden/make_golden.py

What is executed is the unmodified reference: `Sam2MatchingBaselineNoAMG.forward_test`,
`.forward_fill_memory`, `._process_sam_masks`, `MemoryBank.postprocess`, `compute_sim_global_avg`,
`compute_semantic_ios`, `batched_mask_to_box`, `calculate_stability_score` — bound to a light-weight
stand-in for `self` that supplies synthetic tensors at the encoder seams (`_forward_sam`,
`_extract_target_features`, `_forward_encoder`), because the frozen encoders are out of scope and
random-init SAM-2 emits degenerate masks (SURVEY.md §8c).  Intermediate values are captured by wrapping
the functions `forward_test` looks up in its module globals.

Outputs: tests/golden/<case>.npz (inputs are NOT stored — they are regenerated from the seed by
`synth.make_stage_inputs`; a sha256 of the inputs is stored to detect generator drift).
"""
import hashlib
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import ref_shim  # noqa: E402

synth = importlib.import_module("no-time-to-train_b200.synth")

# name -> (n, c, n_cls, shots, ori_hw, seed, degenerate, num_out_instance, clustered)
STAGE_CASES = {
    "stage_a_1024_degenerate": (64, 384, 5, 2, (1024, 1024), 101, True, 10, True),
    "stage_b_480x640": (48, 384, 5, 2, (480, 640), 102, False, 10, True),
    "stage_c_427x640_degenerate": (48, 384, 4, 3, (427, 640), 103, True, 10, True),
    "stage_d_200x180_downscale": (40, 384, 5, 2, (200, 180), 104, False, 10, True),
    "stage_e_config1_1cls_1shot": (100, 384, 1, 1, (1024, 1024), 105, True, 100, False),
    "stage_f_truncate_333x500": (96, 64, 3, 2, (333, 500), 106, False, 4, True),
    "stage_g_iid_80cls": (128, 256, 80, 10, (512, 512), 107, True, 100, False),
    # degenerate == 2: + masks cut by exactly one image border (bottom only, corners, ragged bottom edge)
    "stage_h_borders_640x480": (48, 128, 5, 2, (640, 480), 108, 2, 48, True),
    "stage_i_borders_1024": (32, 64, 3, 2, (1024, 1024), 109, 2, 32, True),
}

# negative-reference cases: name -> (n, c, n_cls, shots_neg, ori_hw, seed, num_out[, degenerate])
# degenerate: the reference's negative path has NO zero guard (matching_baseline_utils.py:925): the empty low-res
# mask of `inject_degenerate_cases` gives a NaN feature row, NaN similarities and a top-k over an all-NaN row.
NEG_CASES = {
    "stageneg_a_5cls_3neg": (64, 384, 5, 3, (480, 640), 301, 10),
    "stageneg_b_20cls_2neg": (96, 256, 20, 2, (512, 512), 302, 20),
    "stageneg_c_degenerate_80cls": (64, 128, 80, 2, (480, 640), 303, 64, 1),
    "stageneg_d_degenerate_borders": (48, 384, 40, 3, (427, 640), 304, 48, 2),
}

# candidate-selection cases (real `_forward_sam` over a stand-in predictor that returns synthetic RAW decoder output):
# name -> (points_per_side, testing_point_bs, m, iou_thr, c, n_cls, shots, ori_hw, seed, num_out)
MULTI_CASES = {
    "stagemm_a_64prompts_bs16": (8, 16, 4, 0.5, 128, 5, 2, (480, 640), 401, 10),
    "stagemm_b_100prompts_bs25": (10, 25, 4, 0.8, 64, 3, 2, (512, 512), 402, 8),
}

# name -> (n_cls, shots, filled_per_class, c, seed)
FILL_CASES = {
    "fill_a_3cls_2shot": (3, 2, [2, 2, 1], 32, 201),
    "fill_b_5cls_3shot": (5, 3, [3, 3, 3, 3, 0], 48, 202),
}


def sha(*tensors) -> str:
    h = hashlib.sha256()
    for t in tensors:
        h.update(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes())
    return h.hexdigest()


def run_stage_case(ref, name, spec):
    n, c, n_cls, shots, ori_hw, seed, degenerate, num_out, clustered = spec
    inp = synth.make_stage_inputs(n, c, n_cls, shots, ori_hw, seed=seed, clustered=clustered,
                                  degenerate=int(degenerate))
    model_mod = sys.modules[ref.Model.__module__]
    cap = {}

    def wrap(fn_name, rec):
        orig = getattr(model_mod, fn_name)

        def inner(*a, **k):
            out = orig(*a, **k)
            rec(a, k, out)
            return out
        setattr(model_mod, fn_name, inner)
        return orig

    boxes_calls = []
    origs = {
        "compute_sim_global_avg": wrap("compute_sim_global_avg",
                                       lambda a, k, o: cap.update(sim=o[0].clone(), obj_feats=o[1].clone())),
        "batched_nms": wrap("batched_nms", lambda a, k, o: cap.update(nms_keep_full=o.clone())),
        "compute_semantic_ios": wrap("compute_semantic_ios",
                                     lambda a, k, o: cap.update(ios=o.clone(), full_masks=a[0].clone(),
                                                                labels_sel=a[1].clone())),
        "batched_mask_to_box": wrap("batched_mask_to_box", lambda a, k, o: boxes_calls.append(o.clone())),
    }
    try:
        fake = types.SimpleNamespace()
        fake.predictor = types.SimpleNamespace(device=torch.device("cpu"))
        fake.encoder_h, fake.encoder_w = 37, 37
        fake.cls_num_per_mask = 1
        fake.num_out_instance = num_out
        fake.nms_thr = 0.5
        fake.online_vis = False
        fake.memory_bank = types.SimpleNamespace(feats_ins_avg=inp.feats_ins_avg, n_classes=n_cls)
        fake.sam_transform = lambda x: x
        fake._extract_target_features = lambda img, device: (inp.tar_feat, img)
        fake._forward_sam = lambda imgs: (inp.lr_masks, inp.pred_ious, None)
        fake._process_sam_masks = types.MethodType(ref.Model._process_sam_masks, fake)
        fake._reset = lambda: None
        info = dict(ori_height=ori_hw[0], ori_width=ori_hw[1], file_name="synthetic", id=0)
        with torch.inference_mode():
            out = ref.Model.forward_test(
                fake, [dict(target_img=torch.zeros(3, 8, 8), target_img_info=info)], False)[0]
            stab = ref.calculate_stability_score(inp.lr_masks, 0.0, 1.0)
    finally:
        for k, v in origs.items():
            setattr(model_mod, k, v)

    full = cap.get("full_masks")
    g = dict(
        spec=np.array([n, c, n_cls, shots, ori_hw[0], ori_hw[1], seed, int(degenerate), num_out,
                       int(clustered)], dtype=np.int64),
        inputs_sha=np.array(sha(inp.lr_masks, inp.pred_ious, inp.tar_feat, inp.feats_ins_avg)),
        sim=cap["sim"].numpy(),
        obj_feats=cap["obj_feats"].numpy(),
        lr_boxes=boxes_calls[0].numpy(),
        nms_keep_full=cap["nms_keep_full"].numpy(),
        stability=stab.numpy(),
        out_scores=out["scores"].numpy(),
        out_labels=out["labels"].numpy(),
        out_bboxes=out["bboxes"].numpy(),
        out_masks_packed=np.packbits(out["binary_masks"].numpy().reshape(out["binary_masks"].shape[0], -1),
                                     axis=-1),
    )
    if full is not None:
        g.update(
            ios=cap["ios"].numpy(),
            labels_sel=cap["labels_sel"].numpy(),
            full_area=full.reshape(full.shape[0], -1).sum(-1).numpy(),
            full_boxes=boxes_calls[1].numpy(),
            full_masks_sha=np.array(sha(full)),
        )
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **g)
    print(f"{name}: K_sel={0 if full is None else full.shape[0]} K_out={out['scores'].shape[0]} "
          f"nan_scores={int(torch.isnan(out['scores']).sum())} labels_used={len(set(out['labels'].tolist()))}")


def run_neg_case(ref, name, spec):
    """forward_test(with_negative=True): needs memory_bank.feats_avg and memory_bank_neg.feats_ins_avg."""
    n, c, n_cls, l_neg, ori_hw, seed, num_out = spec[:7]
    degenerate = spec[7] if len(spec) > 7 else 0
    inp = synth.make_stage_inputs(n, c, n_cls, 2, ori_hw, seed=seed, clustered=True, degenerate=degenerate)
    gen = torch.Generator().manual_seed(seed + 7)
    feats_avg = inp.feats_ins_avg.mean(dim=1) * 3.0  # un-normalised class averages
    neg = inp.feats_ins_avg[:, :1].repeat(1, l_neg, 1) * 0.5 + 0.6 * torch.randn(n_cls, l_neg, c, generator=gen) / (c ** 0.5)
    model_mod = sys.modules[ref.Model.__module__]
    cap = {}
    orig = model_mod.compute_sim_global_avg_with_neg

    def rec(*a, **k):
        out = orig(*a, **k)
        cap["sim"] = out.clone()
        return out
    orig_nms = model_mod.batched_nms

    def rec_nms(*a, **k):
        out = orig_nms(*a, **k)
        cap["nms_keep_full"], cap["labels_all"] = out.clone(), a[2].clone()
        return out
    model_mod.compute_sim_global_avg_with_neg = rec
    model_mod.batched_nms = rec_nms
    try:
        fake = types.SimpleNamespace()
        fake.predictor = types.SimpleNamespace(device=torch.device("cpu"))
        fake.encoder_h, fake.encoder_w = 37, 37
        fake.cls_num_per_mask = 1
        fake.num_out_instance = num_out
        fake.nms_thr = 0.5
        fake.online_vis = False
        fake.memory_bank = types.SimpleNamespace(feats_avg=feats_avg, feats_ins_avg=inp.feats_ins_avg, n_classes=n_cls)
        fake.memory_bank_neg = types.SimpleNamespace(feats_ins_avg=neg)
        fake.sam_transform = lambda x: x
        fake._extract_target_features = lambda img, device: (inp.tar_feat, img)
        fake._forward_sam = lambda imgs: (inp.lr_masks, inp.pred_ious, None)
        fake._process_sam_masks = types.MethodType(ref.Model._process_sam_masks, fake)
        fake._reset = lambda: None
        info = dict(ori_height=ori_hw[0], ori_width=ori_hw[1], file_name="synthetic", id=0)
        with torch.inference_mode():
            out = ref.Model.forward_test(fake, [dict(target_img=torch.zeros(3, 8, 8), target_img_info=info)], True)[0]
    finally:
        model_mod.compute_sim_global_avg_with_neg = orig
        model_mod.batched_nms = orig_nms
    extra = {}
    if degenerate:  # (kept out of the two older files so that they regenerate byte-identically)
        extra = dict(nms_keep_full=cap["nms_keep_full"].numpy(), labels_all=cap["labels_all"].numpy())
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), **extra,
        spec=np.array([n, c, n_cls, l_neg, ori_hw[0], ori_hw[1], seed, num_out] + ([degenerate] if degenerate else []),
                      dtype=np.int64),
        feats_avg=feats_avg.numpy(), feats_ins_avg_neg=neg.numpy(),
        inputs_sha=np.array(sha(inp.lr_masks, inp.pred_ious, inp.tar_feat, inp.feats_ins_avg)),
        sim=cap["sim"].numpy(), out_scores=out["scores"].numpy(), out_labels=out["labels"].numpy(),
        out_bboxes=out["bboxes"].numpy(),
        out_masks_packed=np.packbits(out["binary_masks"].numpy().reshape(out["binary_masks"].shape[0], -1), axis=-1))
    print(f"{name}: K_out={out['scores'].shape[0]} labels_used={len(set(out['labels'].tolist()))} "
          f"sim range [{float(cap['sim'].min()):.3f}, {float(cap['sim'].max()):.3f}]")


def run_multimask_case(ref, name, spec):
    """The reference's own `_forward_sam` (+ `_compute_masks`, `_forward_sam_decoder`: best-of-3 gather, cat,
    `> iou_thr`) over a stand-in predictor whose decoder returns seeded synthetic multimask logits, followed by the
    real `forward_test`."""
    pps, bs, m, iou_thr, c, n_cls, shots, ori_hw, seed, num_out = spec
    n = pps * pps
    multi, ious = synth.make_multimask_inputs(n, m, seed=seed)
    feat_in = synth.make_stage_inputs(8, c, n_cls, shots, ori_hw, seed=seed + 1, clustered=True)
    calls = {"i": 0}

    def decoder(**kw):
        assert kw["multimask_output"] is True and kw["output_all_masks"] is True and kw["repeat_image"] is False
        i = calls["i"]
        calls["i"] += 1
        return multi[i * bs:(i + 1) * bs], ious[i * bs:(i + 1) * bs], None, None

    prompt_encoder = lambda points, boxes, masks: (torch.zeros(bs, 2, 4), torch.zeros(bs, 4, 2, 2))
    prompt_encoder.get_dense_pe = lambda: torch.zeros(1, 4, 2, 2)
    pred = types.SimpleNamespace(
        device=torch.device("cpu"),
        forward_image=lambda imgs: {},
        _prepare_backbone_features=lambda bo: (None, [torch.zeros(16, 1, 4), torch.zeros(4, 1, 4)], None, [(4, 4), (2, 2)]),
        sam_prompt_encoder=prompt_encoder, sam_mask_decoder=decoder)
    cap = {}
    fake = types.SimpleNamespace()
    fake.predictor = pred
    fake.points_per_side, fake.testing_point_bs, fake.iou_thr = pps, bs, iou_thr
    fake.backbone_features = fake.backbone_hr_features = None
    fake._get_grid_points = types.MethodType(ref.Model._get_grid_points, fake)
    fake._compute_masks = types.MethodType(ref.Model._compute_masks, fake)
    fake._forward_sam_decoder = types.MethodType(ref.Model._forward_sam_decoder, fake)
    real_forward_sam = types.MethodType(ref.Model._forward_sam, fake)

    def forward_sam(imgs):
        out = real_forward_sam(imgs)
        cap["lr_masks"], cap["pred_ious"] = out[0].clone(), out[1].clone()
        return out
    fake._forward_sam = forward_sam
    fake.encoder_h, fake.encoder_w = 37, 37
    fake.cls_num_per_mask = 1
    fake.num_out_instance = num_out
    fake.nms_thr = 0.5
    fake.online_vis = False
    fake.memory_bank = types.SimpleNamespace(feats_ins_avg=feat_in.feats_ins_avg, n_classes=n_cls)
    fake.sam_transform = lambda x: x
    fake._extract_target_features = lambda img, device: (feat_in.tar_feat, img)
    fake._process_sam_masks = types.MethodType(ref.Model._process_sam_masks, fake)
    fake._reset = lambda: None
    info = dict(ori_height=ori_hw[0], ori_width=ori_hw[1], file_name="synthetic", id=0)
    with torch.inference_mode():
        out = ref.Model.forward_test(fake, [dict(target_img=torch.zeros(3, 64, 64), target_img_info=info)], False)[0]
    assert calls["i"] == n // bs
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        spec=np.array([pps, bs, m, c, n_cls, shots, ori_hw[0], ori_hw[1], seed, num_out], dtype=np.int64),
        iou_thr=np.array(iou_thr, dtype=np.float64),
        inputs_sha=np.array(sha(multi, ious, feat_in.tar_feat, feat_in.feats_ins_avg)),
        sel_pred_ious=cap["pred_ious"].numpy(), sel_masks_sha=np.array(sha(cap["lr_masks"])),
        sel_count=np.array(cap["lr_masks"].shape[0], dtype=np.int64),
        out_scores=out["scores"].numpy(), out_labels=out["labels"].numpy(), out_bboxes=out["bboxes"].numpy(),
        out_masks_packed=np.packbits(out["binary_masks"].numpy().reshape(out["binary_masks"].shape[0], -1), axis=-1))
    print(f"{name}: prompts={n} kept={cap['lr_masks'].shape[0]} K_out={out['scores'].shape[0]}")


def rle_special_masks():
    """Small masks covering the run-length edge cases: empty, full, first/last pixel set, runs that wrap from the
    bottom of one column into the top of the next, a checkerboard (one run per pixel), widths off the 32-pixel grid."""
    gen = torch.Generator().manual_seed(77)
    out = {}
    out["zeros_9x13"] = torch.zeros(9, 13, dtype=torch.bool)
    out["ones_9x13"] = torch.ones(9, 13, dtype=torch.bool)
    m = torch.zeros(40, 70, dtype=torch.bool); m[0, 0] = True; out["first_pixel"] = m
    m = torch.zeros(40, 70, dtype=torch.bool); m[-1, -1] = True; out["last_pixel"] = m
    m = torch.zeros(64, 96, dtype=torch.bool); m[:, 10:20] = True; m[0:5, 40:45] = True; m[60:, 40:45] = True
    out["column_wrap"] = m
    yy, xx = torch.meshgrid(torch.arange(33), torch.arange(47), indexing="ij")
    out["checker_33x47"] = ((yy + xx) % 2 == 0)
    out["noise_100x75"] = torch.rand(100, 75, generator=gen) > 0.7
    m = torch.zeros(300, 500, dtype=torch.bool); m[20:280, 31:470] = True; m[100:120, 200:260] = False
    out["blob_300x500"] = m
    # masks that reach the LAST row without reaching the first one: the run of a column ends at the bottom border and
    # the next column starts with background, so the closing boundary sits at (x+1, 0), above a tight rect
    m = torch.zeros(64, 96, dtype=torch.bool); m[40:, 10:20] = True; out["bottom_only_block"] = m
    m = torch.zeros(64, 96, dtype=torch.bool); m[50:, 33] = True; out["bottom_only_one_column"] = m
    m = torch.zeros(64, 96, dtype=torch.bool); m[30:, 80:] = True; out["bottom_right_corner"] = m
    m = torch.zeros(64, 96, dtype=torch.bool); m[30:, :12] = True; out["bottom_left_corner"] = m
    m = torch.zeros(70, 130, dtype=torch.bool); m[35:, 20:110] = True; m[60:, 20:110:2] = False
    out["bottom_ragged_multiword"] = m
    m = torch.zeros(64, 96, dtype=torch.bool); m[40:, 31] = True; m[40:, 32] = True; m[20:, 63] = True
    out["bottom_only_word_seams"] = m
    m = torch.zeros(45, 64, dtype=torch.bool); m[10:, 63] = True; out["bottom_only_last_column"] = m
    return out


def run_rle_golden(ref):
    """Counts from the reference's own uncompressed-RLE encoder `mask_to_rle_pytorch` (sam2/utils/amg.py:111-140),
    "in the format expected by pycoco tools": on the special masks and on the output masks of the stage cases."""
    amg = importlib.import_module("sam2.utils.amg")
    store = {}
    for name, m in rle_special_masks().items():
        rle = amg.mask_to_rle_pytorch(m[None])[0]
        assert np.array_equal(amg.rle_to_mask(rle), m.numpy())
        store["special__" + name + "__mask"] = np.packbits(m.numpy().reshape(-1))
        store["special__" + name + "__hw"] = np.array(m.shape, dtype=np.int64)
        store["special__" + name + "__counts"] = np.array(rle["counts"], dtype=np.int64)
    for case in ("stage_a_1024_degenerate", "stage_b_480x640", "stage_f_truncate_333x500", "stage_d_200x180_downscale",
                 "stage_h_borders_640x480", "stage_i_borders_1024"):
        g = np.load(os.path.join(HERE, case + ".npz"))
        oh, ow = int(g["spec"][4]), int(g["spec"][5])
        k = g["out_masks_packed"].shape[0]
        masks = np.unpackbits(g["out_masks_packed"], axis=-1)[:, :oh * ow].reshape(k, oh, ow).astype(bool)
        rles = amg.mask_to_rle_pytorch(torch.from_numpy(masks))
        flat = np.concatenate([np.array(r["counts"], dtype=np.int64) for r in rles]) if k else np.zeros(0, np.int64)
        store["stage__" + case + "__counts"] = flat
        store["stage__" + case + "__lens"] = np.array([len(r["counts"]) for r in rles], dtype=np.int64)
        print(f"rle {case}: {k} masks, {flat.size} counts")
    np.savez_compressed(os.path.join(HERE, "rle_counts.npz"), **store)


def run_fill_case(ref, name, spec):
    n_cls, shots, filled, c, seed = spec
    e_side, img_side = 37, 74
    e = e_side * e_side
    feats, _ = synth.make_ref_shots(n_cls, shots, e, c, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    bank = ref.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(e, c)), 2, 2)
    order = [(ci, li) for li in range(shots) for ci in range(n_cls) if li < filled[ci]]
    calls = {"i": 0}

    def fake_encoder(imgs):
        ci, li = order[calls["i"]]
        calls["i"] += 1
        return feats[ci, li].reshape(1, e, c)

    fake = types.SimpleNamespace()
    fake.predictor = types.SimpleNamespace(device=torch.device("cpu"))
    fake.encoder_img_size = img_side
    fake.encoder_transform = lambda x: x
    fake.encoder_dim = c
    fake.encoder_h, fake.encoder_w = e_side, e_side
    fake._forward_encoder = fake_encoder
    fake.memory_bank = bank
    fake.memory_bank_neg = None
    soft_masks = []
    for ci, li in order:
        m = torch.zeros(1, img_side, img_side)
        y0, x0 = torch.randint(0, img_side // 2, (2,), generator=gen).tolist()
        hh, ww = torch.randint(6, img_side // 2, (2,), generator=gen).tolist()
        m[0, y0:y0 + hh, x0:x0 + ww] = 1.0
        m[0, y0:y0 + 3, x0:x0 + ww] = torch.rand(3, ww, generator=gen)
        soft_masks.append(m)
        img = torch.rand(1, 3, img_side, img_side, generator=gen)
        ref.Model.forward_fill_memory(fake, [dict(refs_by_cat={ci: dict(imgs=img, masks=m)})], True)
    masks_lowres = bank.masks.clone()
    bank.postprocess()
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        spec=np.array([n_cls, shots, c, seed, e_side, img_side], dtype=np.int64),
        filled=np.array(filled, dtype=np.int64),
        order=np.array(order, dtype=np.int64),
        soft_masks=torch.cat(soft_masks).numpy(),
        masks_lowres=masks_lowres.numpy(),
        fill_counts=bank.fill_counts.numpy(),
        feats_avg=bank.feats_avg.numpy(),
        feats_ins_avg=bank.feats_ins_avg.numpy(),
        postprocessed=bank.postprocessed.numpy(),
    )
    print(f"{name}: fill_counts={bank.fill_counts.tolist()}")


def run_target_feature_case(ref, name="target_features_dinov2_s", n_rows=48):
    """The reference's `_extract_target_features` (bicubic 1024 -> 518, ImageNet normalisation, encoder, CLS dropped) on
    the random-init DINOv2 of `sam2_builder.build_dinov2()` and a seeded image: a seeded sample of `n_rows` of its
    [1369, C] output, and the sha256 of the whole output."""
    import sam2_builder
    from torchvision.transforms import Normalize
    enc = sam2_builder.build_dinov2()
    gen = torch.Generator().manual_seed(3)
    img = torch.rand(3, 1024, 1024, generator=gen)
    fake = types.SimpleNamespace(encoder=enc, encoder_img_size=518, encoder_dim=384,
                                 encoder_transform=Normalize(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)))
    for fn in ("_forward_encoder", "_extract_target_features"):
        setattr(fake, fn, types.MethodType(getattr(ref.Model, fn), fake))
    with torch.inference_mode():
        want = fake._extract_target_features(img, torch.device("cpu"))
    want = (want[0] if isinstance(want, tuple) else want).reshape(-1, 384).contiguous()
    rows = np.sort(np.random.default_rng(3).choice(want.shape[0], n_rows, replace=False))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), rows=rows, feat_rows=want[rows].numpy(),
                        shape=np.array(want.shape), feat_sha=sha(want), image_sha=sha(img))
    print(f"{name}: {tuple(want.shape)}, {n_rows} rows stored")


def main():
    torch.manual_seed(0)
    ref = ref_shim.load()
    only = sys.argv[1:]
    for name, spec in STAGE_CASES.items():
        if not only or name in only:
            run_stage_case(ref, name, spec)
    for name, spec in FILL_CASES.items():
        if not only or name in only:
            run_fill_case(ref, name, spec)
    for name, spec in NEG_CASES.items():
        if not only or name in only:
            run_neg_case(ref, name, spec)
    for name, spec in MULTI_CASES.items():
        if not only or name in only:
            run_multimask_case(ref, name, spec)
    if not only or "rle" in only:
        run_rle_golden(ref)
    if not only or "target_features" in only:
        run_target_feature_case(ref)


if __name__ == "__main__":
    main()
