"""The SAM-2 prompting glue of the drop-in class, executed against the REAL reference on the same random-init weights
(BASELINE.json configs[0]: sam2_hiera_t + DINOv2 ViT-S/14 random-init, CPU).

`model._sam2_grid_masks` restates `_forward_sam` / `_compute_masks` / `_forward_sam_decoder`
(`Sam2MatchingBaseline_noAMG.py:259-299, 355-433`) up to — but not including — the best-of-3 gather, the `cat` and the
`iou_thr` compaction, which the stage fuses.  The grid-prompting test drives the original's own SAM-2 predictor and
needs the original no-time-to-train source tree (found through NTTT_REFERENCE_ROOT, see tests/golden/ref_shim.py): it
is skipped without it.  The target-feature test compares with a stored sample of the original's output everywhere, and
with the original itself where that tree is present."""
import hashlib
import importlib
import os
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import ref_shim  # noqa: E402

needs_reference = pytest.mark.skipif(not ref_shim.reference_available(),
                                     reason="needs the original no-time-to-train source tree (NTTT_REFERENCE_ROOT)")


@pytest.fixture(scope="module")
def encoder_and_image():
    """Random-init DINOv2 ViT-S (transformers only) and the seeded test image; no SAM-2 needed."""
    import sam2_builder
    enc = sam2_builder.build_dinov2()
    img = torch.rand(3, 1024, 1024, generator=torch.Generator().manual_seed(3))
    return enc, img


@pytest.fixture(scope="module")
def setup(encoder_and_image):
    import sam2_builder
    ref = ref_shim.load()
    pred = sam2_builder.build_predictor("sam2_hiera_t.yaml")
    return (ref, pred, *encoder_and_image)


def _reference_self(ref, pred, enc, pps, bs, iou_thr):
    fake = types.SimpleNamespace(predictor=pred, points_per_side=pps, testing_point_bs=bs, iou_thr=iou_thr,
                                 backbone_features=None, backbone_hr_features=None, encoder=enc, encoder_dim=384,
                                 encoder_img_size=518)
    for name in ("_get_grid_points", "_compute_masks", "_forward_sam_decoder", "_forward_sam", "_forward_encoder",
                 "_extract_target_features"):
        setattr(fake, name, types.MethodType(getattr(ref.Model, name), fake))
    from torchvision.transforms import Normalize
    fake.encoder_transform = Normalize(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    fake.sam_transform = fake.encoder_transform
    return fake


@needs_reference
@pytest.mark.parametrize("pps,bs", [(10, 25), (6, 12)])
def test_grid_prompting_glue_matches_reference_forward_sam(setup, pps, bs):
    ref, pred, enc, img = setup
    model_mod = importlib.import_module("no-time-to-train_b200.model")
    from oracle import ref_torch
    sam_in = model_mod._normalize(img.unsqueeze(0))
    with torch.inference_mode():
        ours = types.SimpleNamespace(predictor=pred, points_per_side=pps, testing_point_bs=bs)
        chunks, ious, points = model_mod._sam2_grid_masks(ours, sam_in)
        assert len(chunks) == (pps * pps) // bs and tuple(chunks[0].shape) == (bs, 4, 256, 256)
        assert tuple(ious.shape) == (len(chunks) * bs, 4)
        # random-init IoU heads sit near sigmoid(0): place the threshold inside the observed range so that the
        # compaction keeps some prompts and drops others
        best = torch.cat([c for c in ious.split(bs)]).gather(1, (ious[:, 1:].argmax(1) + 1)[:, None]).flatten()
        iou_thr = float(best.median())
        fake = _reference_self(ref, pred, enc, pps, bs, iou_thr)
        want_masks, want_scores, want_points = fake._forward_sam(fake.sam_transform(img.unsqueeze(0)))
        got_masks, got_scores, kept = ref_torch.select_candidates(chunks, list(ious.split(bs)), iou_thr)
    assert 0 < want_masks.shape[0] < len(chunks) * bs
    assert torch.equal(got_scores, want_scores)
    assert torch.equal(got_masks, want_masks)
    assert torch.equal(points[:len(chunks) * bs][kept], want_points)


def test_target_feature_seam_matches_reference(encoder_and_image):
    """`_extract_target_features` (bicubic 1024 -> 518, ImageNet normalisation, encoder, CLS dropped; :511-532).

    tests/golden/target_features_dinov2_s.npz holds 48 seeded rows of the [1369, 384] output on this encoder and image
    and a sha256 of the whole output.  They were recorded from this seam, which is unchanged since it last matched the
    original's `_extract_target_features` bit for bit in the live comparison below; `make_golden.py target_features`
    writes the same file from the original itself."""
    enc, img = encoder_and_image
    model_mod = importlib.import_module("no-time-to-train_b200.model")
    ours = types.SimpleNamespace(encoder=enc, encoder_img_size=518, encoder_dim=384)
    ours._forward_encoder = types.MethodType(model_mod.Sam2MatchingBaselineNoAMG._forward_encoder, ours)
    with torch.inference_mode():
        got = model_mod.Sam2MatchingBaselineNoAMG._extract_target_features(ours, img, torch.device("cpu"))
    assert tuple(got[0].shape) == (1369, 384)
    g = np.load(os.path.join(HERE, "golden", "target_features_dinov2_s.npz"))
    assert hashlib.sha256(img.numpy().tobytes()).hexdigest() == str(g["image_sha"]), "seeded image drifted"
    rows = torch.from_numpy(g["rows"])
    assert torch.equal(got[0][rows], torch.from_numpy(g["feat_rows"]))
    assert hashlib.sha256(got[0].contiguous().numpy().tobytes()).hexdigest() == str(g["feat_sha"])
    if ref_shim.reference_available():
        fake = _reference_self(ref_shim.load(), None, enc, 4, 4, 0.0)
        with torch.inference_mode():
            want = fake._extract_target_features(img, torch.device("cpu"))
        want_feat = want[0] if isinstance(want, tuple) else want
        assert torch.equal(got[0], want_feat.reshape(-1, 384))
