"""The invariant behind the resize's two-tap path.  The library packs two-tap records for an axis only when every span of
it has xsize <= 2, and evaluates each span with two taps there.  The CPU tests run the fp32 recipe of the antialias
tables (the C oracle's orc_aa_weights, every operation individually rounded): from the 256-pixel SAM-2 logits every
up-scaling qualifies, and wherever a three-tap table holds a third weight it is 0, so the terms the two-tap path drops
were fma(0, 0, acc).  Some other up-scalings (96 -> 608, ...) have a three-sample span whose third weight is 0 but
whose sample still enters aten's sum (an inf or NaN there makes the output NaN); the GPU test pins that the library
reproduces that on such a size."""
import importlib

import numpy as np
import pytest
import torch

from oracle import nttt_oracle as orc

DEV = "cuda:0"


def _spans(in_size, out_size):
    xmin, xsize, w = orc.aa_weights(in_size, out_size)
    assert w.shape[1] == 3, (in_size, out_size, w.shape)  # every up-scaling gets a three-tap table
    assert xsize.min() >= 1 and xmin.min() >= 0 and np.all(xmin + xsize <= in_size), (in_size, out_size)
    assert np.all(w[:, 2] == 0), (in_size, out_size)
    assert np.all(w[xsize < 2, 1] == 0), (in_size, out_size)  # the packed w1 of a one-sample span
    return xsize


def test_two_taps_from_256_to_every_size_up_to_8192():
    for out_size in range(257, 8193):
        assert _spans(256, out_size).max() <= 2, out_size
    assert _spans(256, 256).max() <= 2


@pytest.mark.parametrize("in_size", [1, 2, 3, 7, 32, 64, 96, 100, 128, 160, 180, 200, 255, 257, 333, 500, 512, 1000, 1024])
def test_third_weight_is_zero_on_other_input_sizes(in_size):
    rng = np.random.default_rng(in_size)
    outs = {in_size, in_size + 1, 2 * in_size, 4 * in_size, 8192}
    outs.update(int(v) for v in rng.integers(in_size, 8193, size=200))
    for out_size in sorted(outs):
        assert _spans(in_size, out_size).max() <= 3, (in_size, out_size)


def test_some_up_scalings_have_a_three_sample_span():
    for in_size, out_size in [(3, 37), (3, 363), (96, 608), (160, 736)]:
        assert _spans(in_size, out_size).max() == 3, (in_size, out_size)


@pytest.mark.gpu
@pytest.mark.parametrize("lr,ori_hw", [(96, (608, 608)), (160, (736, 736))])
def test_non_finite_logit_under_a_zero_third_weight(lr, ori_hw):
    """A non-finite logit on the zero-weight third sample of a three-sample span makes aten's output NaN (not > 0); a
    two-tap evaluation would ignore it.  Rows and columns of such samples, on otherwise positive masks, bit for bit
    against the oracle."""
    ops = importlib.import_module("no-time-to-train_b200.ops")
    xmin, xsize, _ = orc.aa_weights(lr, ori_hw[0])
    third = [int(xmin[i]) + 2 for i in np.nonzero(xsize == 3)[0]]
    assert third
    gen = torch.Generator().manual_seed(lr)
    logits = torch.ones(6, lr, lr)
    for r in third:
        logits[0, r, :] = float("nan")
        logits[1, r, :] = float("inf")
        logits[2, :, r] = float("nan")
        logits[3, :, r] = float("-inf")
        logits[4, r, r] = float("nan")
    logits[5] = torch.randn(lr, lr, generator=gen) + 0.2
    logits[5, third[0], :] = float("nan")
    d = logits.to(DEV)
    bits, area, box, stab, flags = ops.threshold_pack(d)
    sel = torch.arange(6, dtype=torch.int32, device=DEV)
    n_sel = torch.tensor([6], dtype=torch.int32, device=DEV)
    bits_full, rect, area_full, box_full = ops.upsample_threshold_pack(d, bits, box, flags, sel, n_sel, 6, ori_hw)
    got = ops.unpack_masks(bits_full, rect, n_sel, ori_hw)[:6].cpu().numpy()
    want = orc.aa_resize_threshold(logits.numpy(), ori_hw).astype(bool)
    assert np.array_equal(got, want), f"{(got != want).sum()} pixels differ"
    o_box, o_area = orc.mask_boxes(want.astype(np.uint8))
    assert np.array_equal(area_full.cpu().numpy()[:6], o_area)
    assert np.array_equal(box_full.cpu().numpy()[:6].astype(np.int64), o_box)
