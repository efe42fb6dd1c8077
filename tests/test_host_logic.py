"""CPU tests of the host-side logic: multi-rank memory-bank fill (gloo, world_size 2 and 4), image sharding, checkpoint
intake and the model boundary's argument handling.  The pooling kernels need a GPU, so these tests substitute plain
torch arithmetic for `ops.fill_pool_batch` / `ops.fill_scatter` / `ops.fill_finalize` — the thing under test is the slot
assignment, the single all-reduce and the state-dict contract, not the kernels (those are covered by the `-m gpu`
tests against the reference's golden fill)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_pool_batch(feats, soft_masks, enc_hw, sums, wsums, masks_lowres=None):
    m = torch.nn.functional.interpolate(soft_masks[:, None], size=tuple(enc_hw), mode="nearest").reshape(feats.shape[0], -1)
    sums.copy_((feats * m[..., None]).sum(1))
    wsums.copy_(m.sum(1))
    if masks_lowres is not None:
        masks_lowres.copy_(m)


def _fake_pool_one(feat, soft_mask, enc_hw, sum_slot, wsum_slot, mask_slot=None):
    m = torch.nn.functional.interpolate(soft_mask[None, None], size=tuple(enc_hw), mode="nearest").reshape(-1)
    sum_slot += (feat * m[:, None]).sum(0)
    wsum_slot += m.sum()
    if mask_slot is not None:
        mask_slot += m


def _fake_scatter(sums, wsums, masks_lowres, slot, feats_sum, mask_sum, masks=None):
    fs, ms = feats_sum.view(-1, feats_sum.shape[-1]), mask_sum.view(-1)
    mk = masks.view(-1, masks.shape[-1]) if masks is not None else None
    for i, dst in enumerate(slot.tolist()):
        if dst < 0:
            continue
        fs[dst] += sums[i]
        ms[dst] += wsums[i]
        if mk is not None:
            mk[dst] += masks_lowres[i]


def _fake_finalize(sums, wsum):
    w = wsum.clone()
    w[w == 0] = 1.0
    wall = wsum.sum(1, keepdim=True)
    wall[wall == 0] = 1.0
    return sums / w[..., None], sums.sum(1) / wall


def _patch(monkeypatch):
    """Put the fakes in place of the fill kernels through `monkeypatch`, which undoes them after the test: later tests
    in the same process must reach the CUDA kernels again."""
    ops = importlib.import_module("no-time-to-train_b200.ops")
    monkeypatch.setattr(ops, "fill_pool_batch", _fake_pool_batch)
    monkeypatch.setattr(ops, "fill_pool_accumulate", _fake_pool_one)
    monkeypatch.setattr(ops, "fill_scatter", _fake_scatter)
    monkeypatch.setattr(ops, "fill_finalize", _fake_finalize)


def _shots(n_cls, shots, c):
    synth = importlib.import_module("no-time-to-train_b200.synth")
    return synth.make_ref_shots(n_cls, shots, 1369, c, seed=5)


def _dataset_order(n_cls, shots):
    # COCOMemoryFillDataset emits exactly L consecutive items per category (coco_ref_dataset.py:348-361)
    return [(ci, li) for ci in range(n_cls) for li in range(shots)]


def _worker(rank, world, port, n_cls, shots, c, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _patch(pytest.MonkeyPatch())  # a spawned worker: the patch ends with the process
        pkg = importlib.import_module("no-time-to-train_b200")
        feats, masks = _shots(n_cls, shots, c)
        bank = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
        order = _dataset_order(n_cls, shots)
        # DistributedSampler(shuffle=False): rank r takes items r, r+W, ...; half of them one by one (the model's
        # bs=1 path), the rest as one batch (the runner's batched path)
        mine = order[rank::world]
        half = len(mine) // 2
        for ci, li in mine[:half]:
            bank.fill(ci, feats[ci, li], masks[ci, li].reshape(37, 37), (37, 37))
        rest = mine[half:]
        bank.fill_batch([ci for ci, _ in rest], torch.stack([feats[ci, li] for ci, li in rest]),
                        torch.stack([masks[ci, li].reshape(37, 37) for ci, li in rest]), (37, 37))
        assert bank.fill_counts.sum() == 0 and len(bank._stage_cls) == len(mine)  # staged, not yet slotted
        if rank == 0:
            bank.sync_in_state_dict = False
            with pytest.raises(RuntimeError, match="staged but not yet slotted"):
                bank.state_dict()  # a rank-local state_dict() must not start a collective when told not to
            bank.sync_in_state_dict = True
        sd = bank.state_dict()  # Lightning's save_checkpoint: every rank calls it; the pre-hook resolves the fill
        assert bank.last_sync["allreduce_bytes"] == 4 * n_cls * shots * (c + 1)  # sums + mask sums only
        bank.postprocess()
        torch.save(dict(sd={k: v.clone() for k, v in sd.items()}, ins=bank.feats_ins_avg, avg=bank.feats_avg,
                        counts=bank.fill_counts), os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _single_process_bank(n_cls, shots, c, world, monkeypatch):
    """The same shots through ONE process, in the order the reference's gathered loop sees them with `world` ranks."""
    _patch(monkeypatch)
    pkg = importlib.import_module("no-time-to-train_b200")
    feats, masks = _shots(n_cls, shots, c)
    bank = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    order = _dataset_order(n_cls, shots)
    for step in range(len(order) // world):
        for r in range(world):
            ci, li = order[step * world + r]
            bank.fill(ci, feats[ci, li], masks[ci, li].reshape(37, 37), (37, 37))
    bank.postprocess()
    return bank


@pytest.mark.parametrize("world,n_cls,shots", [(2, 3, 2), (4, 4, 3)])
def test_distributed_fill_matches_single_process_reference(tmp_path, monkeypatch, world, n_cls, shots):
    from oracle import ref_torch
    c = 16
    port = 29500 + (os.getpid() % 2000) + world
    mp.start_processes(_worker, args=(world, port, n_cls, shots, c, str(tmp_path)), nprocs=world, join=True,
                       start_method="spawn")
    feats, masks = _shots(n_cls, shots, c)
    # reference semantics: every rank sees all gathered samples of a step in rank order (:471-485)
    raw = ref_torch.RawBank(n_cls, shots, 1369, c)
    order = _dataset_order(n_cls, shots)
    for step in range(len(order) // world):
        for r in range(world):
            ci, li = order[step * world + r]
            ref_torch.bank_fill(raw, [ci], feats[ci, li][None], masks[ci, li][None])
    want_avg, want_ins = ref_torch.bank_postprocess(raw)
    outs = [torch.load(os.path.join(tmp_path, f"rank{r}.pt")) for r in range(world)]
    single = _single_process_bank(n_cls, shots, c, world, monkeypatch)
    for o in outs:
        assert torch.equal(o["counts"], raw.fill_counts)
        assert torch.equal(o["sd"]["masks"], raw.masks)
        np.testing.assert_allclose(o["ins"].numpy(), want_ins.numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(o["avg"].numpy(), want_avg.numpy(), rtol=1e-5, atol=1e-6)
        # single-writer slots: the all-reduce only adds zeros, so every rank holds exactly what ONE process computes
        assert torch.equal(o["sd"]["feats_sum"], single.feats_sum) and torch.equal(o["sd"]["mask_sum"], single.mask_sum)
        assert torch.equal(o["ins"], single.feats_ins_avg) and torch.equal(o["avg"], single.feats_avg)


def test_single_process_fill_and_state_dict_names(monkeypatch):
    _patch(monkeypatch)
    pkg = importlib.import_module("no-time-to-train_b200")
    n_cls, shots, c = 2, 2, 8
    feats, masks = _shots(n_cls, shots, c)
    bank = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    for ci, li in [(0, 0), (1, 0), (0, 1)]:
        bank.fill(ci, feats[ci, li], masks[ci, li].reshape(37, 37), (37, 37))
    assert bank.fill_counts.tolist() == [2, 1]
    with pytest.raises(IndexError):
        bank.fill(0, feats[0, 0], masks[0, 0].reshape(37, 37), (37, 37))
    bank.postprocess()
    sd = bank.state_dict()
    for k in ("fill_counts", "masks", "feats_avg", "feats_ins_avg", "postprocessed"):
        assert k in sd  # the names the reference checkpoint uses (matching_baseline_utils.py:561-571)
    assert bool(sd["postprocessed"][0])
    # unfilled slot stays zero and takes part in the prototype mean
    assert float(bank.feats_ins_avg[1, 1].abs().max()) == 0.0
    # a reference POST-PROCESSED checkpoint without any of our compact sums loads with strict=False
    ref_sd = {k: v for k, v in sd.items() if k not in ("feats_sum", "mask_sum")}
    other = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    missing, unexpected = other.load_state_dict(ref_sd, strict=False)
    assert set(missing) == {"feats_sum", "mask_sum"} and unexpected == []
    assert torch.equal(other.feats_ins_avg, bank.feats_ins_avg) and bool(other.postprocessed[0])


def test_reference_fill_stage_checkpoint_is_reduced_on_load(monkeypatch):
    """The reference saves after `fill_memory` and post-processes FROM THAT CHECKPOINT (README.md:194-217): its state
    dict holds raw `feats [n_cls, L, E, C]` + `masks` (matching_baseline_utils.py:561-571) and none of our compact sums.
    Loading it must reduce the raw features (sum_e feats * masks) so that `postprocess()` gives what the reference's
    own postprocess gives — not silently leave zero prototypes."""
    from oracle import ref_torch
    _patch(monkeypatch)
    pkg = importlib.import_module("no-time-to-train_b200")
    n_cls, shots, c = 3, 2, 8
    feats, masks = _shots(n_cls, shots, c)
    raw = ref_torch.RawBank(n_cls, shots, 1369, c)
    for ci, li in [(0, 0), (1, 0), (2, 0), (0, 1), (2, 1)]:  # class 1 keeps an unfilled slot
        ref_torch.bank_fill(raw, [ci], feats[ci, li][None], masks[ci, li][None])
    want_avg, want_ins = ref_torch.bank_postprocess(raw)
    # the reference's fill-stage state dict (zeros for everything post-process would write)
    ref_sd = {"fill_counts": raw.fill_counts, "feats": raw.feats, "masks": raw.masks,
              "feats_avg": torch.zeros(n_cls, c), "feats_ins_avg": torch.zeros(n_cls, shots, c),
              "feats_covariances": torch.zeros(n_cls, c, c), "feats_centers": torch.zeros(n_cls, 2, c),
              "ins_sim_avg": torch.zeros(n_cls), "pca_mean": torch.zeros(n_cls, c),
              "pca_components": torch.zeros(n_cls, 2, c), "postprocessed": torch.zeros(1, dtype=torch.bool)}
    bank = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    missing, unexpected = bank.load_state_dict(ref_sd, strict=False)
    assert "feats" not in unexpected and "feats_sum" not in missing and "mask_sum" not in missing
    assert set(unexpected) == {"feats_covariances", "feats_centers", "ins_sim_avg", "pca_mean", "pca_components"}
    assert bank.fill_counts.tolist() == raw.fill_counts.tolist() and not bool(bank.postprocessed[0])
    bank.postprocess()
    np.testing.assert_allclose(bank.feats_ins_avg.numpy(), want_ins.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(bank.feats_avg.numpy(), want_avg.numpy(), rtol=1e-5, atol=1e-6)
    assert float(bank.feats_ins_avg[1, 1].abs().max()) == 0.0
    # the same through a parent module with the reference's key prefix, as the Lightning checkpoint nests it
    holder = torch.nn.Module()
    holder.memory_bank = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    holder.load_state_dict({"memory_bank." + k: v for k, v in ref_sd.items()}, strict=False)
    assert torch.equal(holder.memory_bank.feats_sum, bank.feats_sum)
    # wrong raw shape -> a load error, not a silent skip
    bad = dict(ref_sd, feats=torch.zeros(n_cls, shots, 4, c))
    with pytest.raises(RuntimeError, match="feats has shape"):
        pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c))).load_state_dict(bad, strict=False)
    # a state dict with masks but neither sums nor raw feats: postprocess refuses instead of writing zero prototypes
    lost = {k: v for k, v in ref_sd.items() if k != "feats"}
    broken = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(1369, c)))
    broken.load_state_dict(lost, strict=False)
    with pytest.raises(RuntimeError, match="inconsistent"):
        broken.postprocess()


def test_image_sharding_is_strided_and_complete():
    """Test-time sharding mirrors DistributedSampler(shuffle=False) + the re-interleave of
    collect_results_cpu (run_lightning.py:69-75)."""
    shard = importlib.import_module("no-time-to-train_b200.sharding")
    for n, w in [(256, 8), (10, 4), (7, 2), (3, 4)]:
        parts = [shard.shard_indices(n, r, w) for r in range(w)]
        assert len({len(p) for p in parts}) == 1  # padded to equal length by repetition
        merged = shard.interleave([[f"img{i}" for i in p] for p in parts], n)
        assert merged == [f"img{i}" for i in range(n)]


def _collect_worker(rank, world, port, n_items, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        shard = importlib.import_module("no-time-to-train_b200.sharding")
        # each rank "scores" its images: one encoded-result list per image, as `_output_inqueue` appends them
        part = [[dict(image_id=i, category_id=7, score=0.5, segmentation=dict(size=[4, 4], counts="`0"))]
                for i in shard.shard_indices(n_items, rank, world)]
        got = shard.collect_results(part, size=n_items)
        torch.save(got, os.path.join(out_dir, f"collect{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_collect_results_gathers_and_reorders(tmp_path):
    """`collect_results` == the reference's `collect_results_cpu` (run_lightning.py:23-78): rank 0 gets every image's
    results in dataset order, truncated to the dataset length (7 images on 2 ranks: one padded repeat); other
    ranks get None; without a process group the part comes back unchanged."""
    shard = importlib.import_module("no-time-to-train_b200.sharding")
    assert shard.collect_results([1, 2, 3], size=2) == [1, 2, 3]
    n_items, world = 7, 2
    port = 31500 + (os.getpid() % 2000)
    mp.start_processes(_collect_worker, args=(world, port, n_items, str(tmp_path)), nprocs=world, join=True,
                       start_method="spawn")
    got0 = torch.load(os.path.join(tmp_path, "collect0.pt"))
    got1 = torch.load(os.path.join(tmp_path, "collect1.pt"))
    assert got1 is None
    assert [r[0]["image_id"] for r in got0] == list(range(n_items))


def test_model_rejects_unsupported_modes_without_gpu():
    pkg = importlib.import_module("no-time-to-train_b200")
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.Sam2MatchingBaselineNoAMG(sam2_infer_cfgs=dict(nms_thr=0.5, num_out_instance=10, cls_num_per_mask=1),
                                      memory_bank_cfg=dict(enable=True, category_num=2, length=1),
                                      encoder_geometry=(518, 14, 8))
