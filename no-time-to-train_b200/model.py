"""Drop-in mirror of the reference's matching model for the reference-matching stage.

`Sam2MatchingBaselineNoAMG` keeps the reference's boundary
(`no_time_to_train/models/Sam2MatchingBaseline_noAMG.py:128-765`): same constructor keywords, same
`forward(input_dicts)` with `data_mode` in {fill_memory, test, ...}, same `postprocess_memory()`, same
`memory_bank.*` buffers in the state dict, same output dict and the same errors.  It is what
`Sam2MatcherLightningModel` (`pl_wrapper/sam2matcher_pl.py:131-135, 163-201`) instantiates and calls.

Everything between the encoder seams and the output dict runs in libnttt_b200.so (hand-written sm_100a CUDA
behind the C-ABI of include/nttt_b200.h).  The frozen encoders stay ordinary PyTorch modules and are injected:
`predictor` (a SAM-2 `SAM2VideoPredictor`) and `encoder` (a HF DINOv2/DINOv3 `AutoModel`) are built with the
reference's own builders when its packages are importable, or passed in by the caller (tests and the
benchmark pass seam objects that emit synthetic tensors, SURVEY.md §8d).
"""
from __future__ import annotations

import copy

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .matching import MatchingStage, StageConfig
from .memory_bank import MemoryBank

_IMAGENET_MEAN = (0.485, 0.456, 0.406)
_IMAGENET_STD = (0.229, 0.224, 0.225)

# encoder presets: (img_size, patch_size) per `encoder_cfg` key (reference table at
# Sam2MatchingBaseline_noAMG.py:26-126; only the geometry is needed here)
ENCODER_GEOMETRY = {
    "dinov2_small": (518, 14), "dinov2_base": (518, 14), "dinov2_large": (518, 14), "dinov2_giant": (518, 14),
}


def _normalize(x, mean=_IMAGENET_MEAN, std=_IMAGENET_STD):
    m = torch.tensor(mean, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
    s = torch.tensor(std, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
    return (x - m) / s


class Sam2MatchingBaselineNoAMG(nn.Module):
    def __init__(self, sam2_cfg_file=None, sam2_ckpt_path=None, sam2_infer_cfgs=None, encoder_cfg=None,
                 encoder_ckpt_path=None, memory_bank_cfg=None, dataset_name="coco", dataset_imgs_path=None,
                 class_names=None, online_vis=False, vis_thr=0.5, *, predictor=None, encoder=None,
                 encoder_geometry=None, device=None):
        super().__init__()
        sam2_infer_cfgs = dict(sam2_infer_cfgs or {})
        memory_bank_cfg = dict(memory_bank_cfg or {})
        self.dataset_name = dataset_name
        self.class_names = class_names
        self.dataset_imgs_path = dataset_imgs_path
        self.online_vis = online_vis
        self.vis_thr = vis_thr
        self.points_per_side = sam2_infer_cfgs.get("points_per_side")
        self.testing_point_bs = sam2_infer_cfgs.get("testing_point_bs")
        self.iou_thr = sam2_infer_cfgs.get("iou_thr")
        self.num_out_instance = sam2_infer_cfgs.get("num_out_instance")
        self.nms_thr = sam2_infer_cfgs.get("nms_thr")
        self.kmeans_k = sam2_infer_cfgs.get("kmeans_k")
        self.n_pca_components = sam2_infer_cfgs.get("n_pca_components")
        self.cls_num_per_mask = sam2_infer_cfgs.get("cls_num_per_mask")
        self.with_negative_refs = sam2_infer_cfgs.get("with_negative_refs", False)

        if device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("Sam2MatchingBaselineNoAMG (B200) needs a CUDA device; there is no CPU path")
            device = torch.device("cuda", torch.cuda.current_device())
        self._device = torch.device(device)

        if predictor is None and sam2_cfg_file is not None:
            predictor = _build_reference_predictor(sam2_cfg_file, sam2_ckpt_path, self._device)
        self.predictor = predictor
        self.sam_img_size = 1024
        if encoder is None and encoder_cfg is not None and encoder_geometry is None:
            encoder, encoder_geometry = _build_reference_encoder(encoder_cfg, encoder_ckpt_path, self._device)
        self.encoder = encoder
        if encoder_geometry is None:
            raise ValueError("encoder_geometry=(img_size, patch_size, hidden_size) is required with an injected encoder")
        self.encoder_img_size, self.encoder_patch_size, self.encoder_dim = encoder_geometry
        self.encoder_h = self.encoder_w = self.encoder_img_size // self.encoder_patch_size

        assert memory_bank_cfg.pop("enable", True)
        memory_bank_cfg["feat_shape"] = (self.encoder_h * self.encoder_w, self.encoder_dim)
        self.model_cfg_memory = copy.deepcopy(memory_bank_cfg)
        self.memory_bank = MemoryBank(memory_bank_cfg, self.kmeans_k, self.n_pca_components).to(self._device)
        if self.with_negative_refs:  # (:225-230)
            neg_cfg = copy.deepcopy(memory_bank_cfg)
            neg_cfg["length"] = memory_bank_cfg.get("length_negative")
            self.memory_bank_neg = MemoryBank(neg_cfg, self.kmeans_k, self.n_pca_components).to(self._device)
        else:
            self.memory_bank_neg = None

        k = self.cls_num_per_mask
        if k == -1 and self.memory_bank.n_classes == 1:
            k = 1
        self.stage = MatchingStage(self._device, StageConfig(
            nms_thr=float(self.nms_thr), num_out_instance=int(self.num_out_instance), cls_num_per_mask=int(k),
            enc_hw=(self.encoder_h, self.encoder_w)))
        self._proto_version = None
        # Output buffers of forward_test, reused round-robin (see `output_ring`): (ori_hw) -> [ring of (masks, prev_rect)]
        self._out_ring = {}
        self._out_next = {}
        self._reset()
        self.eval()

    # ------------------------------------------------------------------ encoder seams (frozen, as-is PyTorch)
    def _reset(self):
        self.backbone_features = None
        self.backbone_hr_features = None

    def _forward_encoder(self, imgs):
        """Patch tokens of the frozen encoder, CLS/register tokens dropped (:240-257)."""
        n_skip = 1 + getattr(self.encoder.config, "num_register_tokens", 0)
        tokens = self.encoder(pixel_values=imgs, output_hidden_states=False).last_hidden_state
        return tokens[:, n_skip:, :].reshape(imgs.shape[0], -1, self.encoder_dim)

    def _extract_target_features(self, tar_img, device):
        """(:511-532) bicubic resize to the encoder size, ImageNet normalisation, encoder forward."""
        tar_img = tar_img.to(device=device)
        x = F.interpolate(tar_img.unsqueeze(0), size=(self.encoder_img_size, self.encoder_img_size), mode="bicubic")
        return self._forward_encoder(_normalize(x)).reshape(-1, self.encoder_dim), tar_img

    def _forward_sam_raw(self, imgs):
        """(:355-426) grid-prompted SAM-2 decoding, stopped BEFORE the reference's best-of-3 gather, `cat` and
        `iou_thr` compaction (:295-299, :423-431) — those are fused into the stage (SURVEY.md §8f rank 2).
        Returns the decoder's raw per-batch outputs: chunks (list of [bs,4,256,256]), ious [N,4], points."""
        if self.predictor is None or not hasattr(self.predictor, "forward_image"):
            raise RuntimeError("no SAM-2 predictor was provided")
        return _sam2_grid_masks(self, imgs)

    def _forward_sam(self, imgs):
        """(:355-433) the reference's seam: compacted `lr_masks [N,256,256], pred_ious [N], points`.  `forward_test`
        only goes through it when a subclass overrides it (tests inject synthetic candidates here) or when
        `fuse_candidate_selection` is off; otherwise the raw decoder output is handed to the stage in place."""
        chunks, ious, points = self._forward_sam_raw(imgs)
        multi = torch.cat(chunks, dim=0)
        best = torch.argmax(ious[:, 1:], dim=-1) + 1
        rows = torch.arange(multi.shape[0], device=multi.device)
        masks, scores = multi[rows, best], ious[rows, best]
        keep = scores > self.iou_thr
        return masks[keep], scores[keep], points[:multi.shape[0]][keep]

    fuse_candidate_selection = True
    # forward_test writes its `binary_masks` into a small ring of PERSISTENT buffers per image size instead of a fresh
    # 105 MB allocation per image: only the rectangles that change between two uses of a buffer are rewritten
    # (`nttt_match_args.out_prev_rect`), which removes the stage's largest write.  The tensors of a result therefore
    # stay valid for the next `output_ring - 1` calls — ample for the reference's driver, which converts every result
    # to numpy before the next image (`pl_wrapper/sam2matcher_pl.py:144-158`).  0 = a fresh dense buffer per call.
    output_ring = 4
    # True: forward_test also returns `segmentations` (COCO RLE dicts produced on the device by `nttt_rle_encode`),
    # which is what `_output_inqueue` / `encode_results` turn the masks into on the host in the reference
    # (`pl_wrapper/sam2matcher_pl.py:144-158`, `dataset/coco_ref_dataset.py:590-613`).  Off by default: the output dict
    # then has exactly the reference's keys.
    emit_rle = False

    def _persistent_out(self, ori_hw):
        if self.output_ring <= 0:
            return None
        key = (int(ori_hw[0]), int(ori_hw[1]))
        ring = self._out_ring.get(key)
        if ring is None:
            if len(self._out_ring) >= 8:  # datasets with many image sizes: keep the most recent few
                drop = next(iter(self._out_ring))
                del self._out_ring[drop], self._out_next[drop]
            num_out = max(int(self.num_out_instance), 1)
            ring = [(torch.zeros((num_out, key[0], key[1]), dtype=torch.uint8, device=self._device),
                     torch.zeros((num_out, 4), dtype=torch.int32, device=self._device)) for _ in range(self.output_ring)]
            self._out_ring[key] = ring
            self._out_next[key] = 0
        i = self._out_next[key]
        self._out_next[key] = (i + 1) % len(ring)
        return ring[i]

    # ------------------------------------------------------------------ modes
    def forward_fill_memory(self, input_dicts, is_positive=True):
        """(:435-487) one reference shot: encoder forward, then pooled into its (class, slot)."""
        with torch.inference_mode():
            assert len(input_dicts) == 1
            target_bank = self.memory_bank if is_positive else self.memory_bank_neg
            refs = input_dicts[0]["refs_by_cat"]
            cat_ind = list(refs.keys())[0]
            imgs = refs[cat_ind]["imgs"].to(device=self._device)
            masks = refs[cat_ind]["masks"].to(dtype=imgs.dtype)
            imgs = F.interpolate(imgs, size=(self.encoder_img_size, self.encoder_img_size), mode="bicubic")
            feats = self._forward_encoder(_normalize(imgs)).reshape(1, -1, self.encoder_dim)
            target_bank.fill(int(cat_ind), feats[0].float(), masks[0], (self.encoder_h, self.encoder_w))
            return {}

    def postprocess_memory(self):
        """(:700-704)"""
        self.memory_bank.postprocess()

    def postprocess_memory_negative(self):
        """(:706-710)"""
        self.memory_bank_neg.postprocess()

    def _ensure_prototypes(self, with_negative):
        if with_negative:
            ver = ("neg", self.memory_bank.feats_avg._version, self.memory_bank_neg.feats_ins_avg._version)
            if self._proto_version != ver:
                self.stage.set_prototypes_with_negatives(self.memory_bank.feats_avg, self.memory_bank_neg.feats_ins_avg)
                self._proto_version = ver
        else:
            ver = ("pos", self.memory_bank.feats_ins_avg._version)
            if self._proto_version != ver:
                self.stage.set_prototypes(self.memory_bank.feats_ins_avg)
                self._proto_version = ver

    def forward_test(self, input_dicts, with_negative=False):
        """(:562-698) encoders as-is, then the whole matching stage in one `nttt_match_image` call."""
        assert len(input_dicts) == 1
        device = self._device
        with torch.inference_mode():
            tar_feat, tar_img = self._extract_target_features(input_dicts[0]["target_img"], device)
            info = input_dicts[0]["target_img_info"]
            ori_hw = (info["ori_height"], info["ori_width"])
            self._ensure_prototypes(with_negative)
            sam_in = _normalize(tar_img.unsqueeze(0))
            seam_overridden = type(self)._forward_sam is not Sam2MatchingBaselineNoAMG._forward_sam
            # the fused path hands the stage one address per decoder batch, at most _lib.MAX_CHUNKS of them: a denser
            # grid for its batch size (points_per_side 128 with testing_point_bs 128) takes the compacting seam instead
            if (self.fuse_candidate_selection and not seam_overridden and
                    int(self.points_per_side) ** 2 // int(self.testing_point_bs) <= _lib.MAX_CHUNKS):
                chunks, multi_ious, _ = self._forward_sam_raw(sam_in)
                out = self.stage.match([c.float().contiguous() for c in chunks], None, tar_feat.float().contiguous(),
                                       ori_hw, iou_thr=float(self.iou_thr),
                                       multi_ious=multi_ious.float().contiguous(), multi_first=1,
                                       persistent_out=self._persistent_out(ori_hw), rle=self.emit_rle)
            else:
                lr_masks, pred_ious, _ = self._forward_sam(sam_in)
                out = self.stage.match(lr_masks.float().contiguous(), pred_ious.float().contiguous().reshape(-1),
                                       tar_feat.float().contiguous(), ori_hw,
                                       persistent_out=self._persistent_out(ori_hw), rle=self.emit_rle)
        self._reset()
        result = dict(binary_masks=out["binary_masks"], bboxes=out["bboxes"], scores=out["scores"],
                      labels=out["labels"], image_info=info)
        if self.emit_rle:
            result["segmentations"] = out["segmentations"]
        return [result]

    def forward(self, input_dicts):
        """(:712-765) mode dispatch."""
        data_mode = input_dicts[0].pop("data_mode", None)
        assert data_mode is not None
        assert not self.training
        def ready(bank, what):
            if not bank.ready:
                if bank.postprocessed[0].item():
                    bank.ready = True
                else:
                    raise RuntimeError(what)

        if data_mode == "fill_memory":
            return self.forward_fill_memory(input_dicts, is_positive=True)
        if data_mode == "fill_memory_neg":
            assert self.with_negative_refs
            assert not self.memory_bank_neg.postprocessed[0].item()
            return self.forward_fill_memory(input_dicts, is_positive=False)
        if data_mode == "test":
            ready(self.memory_bank, "Memory is not ready!")
            if self.with_negative_refs:
                ready(self.memory_bank_neg, "Negative memory is not ready!")
                return self.forward_test(input_dicts, with_negative=True)
            return self.forward_test(input_dicts, with_negative=False)
        if data_mode == "test_support":
            assert self.with_negative_refs
            ready(self.memory_bank, "Memory is not ready!")
            assert not self.memory_bank_neg.ready
            assert not self.memory_bank_neg.postprocessed[0].item()
            return self.forward_test(input_dicts, with_negative=False)
        if data_mode == "vis_memory":
            raise NotImplementedError("vis_memory is visualisation, outside the B200 hot-path scope (SURVEY.md §2)")
        raise NotImplementedError(f"Unrecognized data mode during inference: {data_mode}")


# ----------------------------------------------------------------------------------------------------------
# encoder construction / SAM-2 prompting glue — only reachable when the reference's packages are installed
# ----------------------------------------------------------------------------------------------------------
def _build_reference_predictor(cfg_file, ckpt_path, device):
    try:
        from sam2.build_sam import build_sam2_video_predictor
    except Exception as exc:  # hydra / sam2 not installed
        raise RuntimeError("building SAM-2 needs the reference's `sam2` package (and hydra); "
                           "pass predictor=... instead") from exc
    return build_sam2_video_predictor(cfg_file, ckpt_path, device=str(device)).eval()


def _build_reference_encoder(encoder_cfg, ckpt_path, device):
    from transformers import AutoModel
    key = encoder_cfg if isinstance(encoder_cfg, str) else encoder_cfg.get("name")
    img_size, patch = ENCODER_GEOMETRY.get(key, (518, 14))
    enc = AutoModel.from_pretrained(ckpt_path).to(device).eval()
    return enc, (img_size, patch, enc.config.hidden_size)


def _sam2_grid_masks(model, imgs):
    """Grid-point prompting of the frozen SAM-2 decoder (`_forward_sam` / `_compute_masks` / `_forward_sam_decoder`,
    :259-426), encoder-side glue kept in plain PyTorch.  The decoder's raw outputs are returned batch by batch; the
    best-of-3 plane choice, the concatenation and the `pred_iou > iou_thr` filter happen inside the stage."""
    pred = model.predictor
    device = imgs.device
    side = imgs.shape[-2]
    lin = torch.linspace(0, side - 1, model.points_per_side)
    gx, gy = torch.meshgrid(lin, lin, indexing="ij")
    points = (torch.stack((gy.reshape(-1), gx.reshape(-1)), dim=-1) + 0.5).to(device)
    backbone_out = pred.forward_image(imgs)
    _, vis_feats, _, feat_sizes = pred._prepare_backbone_features(backbone_out)
    bs = model.testing_point_bs
    img_feats = vis_feats[-1].permute(1, 2, 0).reshape(1, -1, *feat_sizes[-1]).expand(bs, -1, -1, -1)
    hr_feats = [x.permute(1, 2, 0).reshape(1, -1, *s).expand(bs, -1, -1, -1)
                for x, s in zip(vis_feats[:-1], feat_sizes[:-1])]
    chunks, ious = [], []
    for start in range(0, (points.shape[0] // bs) * bs, bs):
        pts = points[start:start + bs].reshape(bs, 1, 2)
        lbl = torch.ones((bs, 1), dtype=torch.int32, device=device)
        sparse, dense = pred.sam_prompt_encoder(points=(pts, lbl), boxes=None, masks=None)
        multi, iou, _, _ = pred.sam_mask_decoder(  # same keywords as the reference call (:275-288)
            image_embeddings=img_feats, image_pe=pred.sam_prompt_encoder.get_dense_pe(),
            sparse_prompt_embeddings=sparse, dense_prompt_embeddings=dense, multimask_output=True,
            repeat_image=False, high_res_features=hr_feats, return_iou_token_out=False,
            disable_custom_iou_embed=True, disable_mlp_obj_scores=True, output_all_masks=True)
        chunks.append(multi)
        ious.append(iou)
    return chunks, torch.cat(ious, dim=0), points
