"""CPU tests of `bench.py --dump-outputs`: the results of the last timed step are written as float `.npy` files, padded
past each image's n_out, masks sampled only where their stream slot still holds them, within the size budget."""
import importlib
import os

import numpy as np
import torch

import bench

matching = importlib.import_module("no-time-to-train_b200.matching")

NUM_OUT, HW = 3, (4, 5)


def _step(images, n_slots, n_out_of):
    """A fake last step: launch r runs image images[r] on slot r % n_slots and returns n_out_of(r) rows whose values
    depend on r, so an image launched twice returns different results each time; slot mask buffers are shared."""
    slot_masks = [torch.zeros((NUM_OUT, *HW), dtype=torch.uint8) for _ in range(n_slots)]
    step = []
    for r, img in enumerate(images):
        k, n_out = r % n_slots, n_out_of(r)
        slot_masks[k].zero_()
        slot_masks[k][:n_out, :, : r % HW[1] + 1] = 1
        counts = torch.tensor([n_out + 5, n_out + 2 if n_out else 0, n_out, 0], dtype=torch.int32)
        pend = matching.PendingResult(None, slot_masks[k].view(torch.bool),
                                      boxes=torch.arange(NUM_OUT * 4, dtype=torch.int64).reshape(NUM_OUT, 4) + r,
                                      scores=torch.linspace(0.9, 0.1, NUM_OUT) - 0.01 * r,
                                      labels=torch.full((NUM_OUT,), r % 7, dtype=torch.int64),
                                      index=torch.arange(NUM_OUT, dtype=torch.int32) * (r + 1), counts=counts, taps={},
                                      ori_hw=HW, keepalive=None)
        step.append((img, k, pend))
    return step


def test_dump_writes_the_last_step_as_float_arrays(tmp_path):
    n_outs = [3, 1, 0, 2, 3, 2]
    # image 100 runs twice (launches 0 and 4), as when a step holds more images than the rank's shard
    step = _step([100, 101, 102, 103, 100, 104], 2, lambda r: n_outs[r])
    bench.dump_outputs(str(tmp_path), step, NUM_OUT)
    a = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert set(a) == {"image", "counts", "scores", "labels", "bboxes", "index", "mask_image", "mask_area",
                      "mask_samples", "mask_pixels"}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    launches = [1, 2, 3, 4, 5]  # the last launch of every distinct image, in launch order
    assert a["image"].tolist() == [101, 102, 103, 100, 104]
    for j, r in enumerate(launches):
        pend, n_out = step[r][2], n_outs[r]
        assert a["counts"][j].tolist() == [n_out + 5, n_out + 2 if n_out else 0, n_out]
        assert np.array_equal(a["scores"][j, :n_out], pend.scores[:n_out].numpy())
        assert np.array_equal(a["bboxes"][j, :n_out], pend.boxes[:n_out].numpy())
        assert np.array_equal(a["labels"][j, :n_out], pend.labels[:n_out].numpy())
        assert np.array_equal(a["index"][j, :n_out], pend.index[:n_out].numpy())
        assert np.isnan(a["scores"][j, n_out:]).all() and np.isnan(a["bboxes"][j, n_out:]).all()
    # slot 0 last ran launch 4 (image 100), slot 1 launch 5 (image 104): only their masks are still in the buffers
    assert a["mask_image"].tolist() == [100, 104]
    assert a["mask_area"][0].tolist() == [4 * 5] * 3
    assert a["mask_area"][1].tolist()[:2] == [4 * 1, 4 * 1] and np.isnan(a["mask_area"][1, 2])
    pix = a["mask_pixels"].astype(np.int64)
    assert len(pix) == HW[0] * HW[1]
    for j, r in enumerate((4, 5)):
        n_out = n_outs[r]
        full = step[r][2].masks.reshape(NUM_OUT, -1).numpy()
        assert np.array_equal(a["mask_samples"][j, :n_out], full[:n_out, pix].astype(np.float32))
        assert np.isnan(a["mask_samples"][j, n_out:]).all()


def test_dump_keeps_to_its_budget_with_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 2048)
    step = _step(list(range(40)), 4, lambda r: 3)
    first = bench.dump_outputs(str(tmp_path / "a"), step, NUM_OUT)
    again = bench.dump_outputs(str(tmp_path / "b"), step, NUM_OUT)
    assert len(first["image"]) < 40 and len(first["mask_pixels"]) < HW[0] * HW[1]
    assert sum(v.nbytes for v in first.values()) <= 2048
    for name, v in first.items():
        assert np.array_equal(v, again[name], equal_nan=True), name
