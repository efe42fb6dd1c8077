"""Accuracy of the memory-bank fill, its post-processing, the prototypes and the negative-reference scoring against
float64 and exact references, per element.

These kernels build the B operand of the similarity GEMM (csrc/fill.cu, csrc/score.cu).  The golden comparisons
(1e-3 of the matrix maximum) cannot see a lost column strip, a dropped patch, a wrong nearest index or a split-K
partial that is never added; these tests can.  The references live in tests/bank_ref.py.

Metrics and tolerances, set a priori from each kernel's order of operations (Higham's gamma_n = n u / (1 - n u),
u = 2^-24), not from a measurement:
  fill_pool sums    |got - sum64| <= TOL_FILL * sum_e |m_e| |f_e|, TOL_FILL = gamma_{ceil(E/8) + 8}: a column's longest
                    chain is ceil(E/8) fmas in one warp, then the 8 warp partials (1.07e-5 at E = 1369).
  fill_pool wsums   |got - wsum64| <= TOL_WSUM * sum_e |m_e|, TOL_WSUM = gamma_{ceil(E/32) + 5} (per-lane adds, then a
                    5-level butterfly).
  low-res masks, fill_pool_accumulate, fill_scatter, fill_finalize: bit for bit (the same fp32 operations restated).
  proto_prepare     |got - proto64| <= gamma_{shots + ceil(c/32) + 8} * bound, bound_i = (S_i + |p_i| ||S||) / ||m|| +
                    |p_i| with S the mean of |x_l| (bank_ref.proto64): the mean's adds and division, the squared norm's
                    fmas and butterfly, the square root, the final division.  Zero class rows must be exact zeros.
  negative scoring  |got - sim64| <= TOL_SIM * B, TOL_SIM from test_gemm_accuracy.py, B the first-order propagation of
                    the two GEMMs' bounds through sp * exp(-clamp(sn - sp, 0) / sigma) plus the fp32 roundings after
                    them (bank_ref.neg64).
The CPU window tests show on the GPU cases' inputs that these limits admit a correct fp32 sum in another order and
reject the emulated defects by >= 4x: a dropped last patch (where one patch is a large enough share of the sum: E <=
1369), a dropped warp partial, the negative max over all slots but the last, no clamp on sim_pos, sigma multiplied
instead of divided.  Comparing sim_neg with the running max before its clamp is an equivalent mutant (the max starts at
0, so a negative value never wins) and no test can catch it.

Cases and the branch each one reaches (each asserts its branch on the host):
  fill_pool_batch (shots, c, grid, mask):
    (16, 1024, 37x37, 518x518)   the product's geometry: 8 column strips, scale 14
    (5, 1536, 37x37, 480x640)    12 strips, non-square mask, non-integer scales
    (3, 1000, 37x37, 74x74)      vector path with a 104-column tail strip
    (3, 1022, 32x32, 1000x1000)  scalar path (c % 4 != 0), E % 8 == 0
    (2, 66, 24x40, 333x500)      scalar path on a non-square grid
    (2, 384, 74x74, 768x768)     aten's fp32 index differs from exact arithmetic at dst 37 (383 vs 384)
    (1, 64, 37x37, 18x18)        up-scaling
    (1, 64, 32x32, 16x16)        up-scaling through aten's out == 2 in shortcut
    (2, 128, 112x112, 200x200)   dynamic shared memory above 48 KB
    (1, 8, 224x224, 224x224)     shared memory exactly at the 200 KB limit; 225x225 is refused, outputs untouched
  fill_pool_accumulate at c = 1024 and c = 66; fill_scatter with out-of-order and skipped slots, masks given and NULL;
  fill_finalize at 1203 x 10 x 1024 with unfilled slots, an empty class and a tiny non-zero weight;
  proto_prepare at 1203 x 10 x 1024, 80 x 30 x 1536, shots = 1 and c = 100 (not a multiple of 32);
  an 80 x 10 bank at c = 1024, E = 1369 filled shot by shot (accumulate) and in batches of 16 (pool + scatter).
  similarity_neg_top1 (n, c, n_cls, l_neg, sigma), throughput launch (no split-K):
    (1, 384, 1, 1, 0.8)          one class: the k == n_cls rule of the top-1 score
    (128, 100, 9, 5, 0.8)        K padded from 100 to 128
    (129, 1024, 80, 3, 0.8)      240 negative columns
    (513, 1024, 1203, 2, 0.8)    256-wide tiles with an N tail on both GEMMs
    (300, 1536, 80, 1, 0.8)      one negative slot
    (200, 768, 40, 4, 0.05 / 10) steep and flat decay
  stage with negatives (n, c, n_cls, l_neg), throughput with pool_order 1 and 0, and low latency:
    (129, 768, 9, 3)             low latency splits both similarity GEMMs (8 partials each)
    (1024, 1024, 80, 3)          ordered pooling at the product's size; split-K on both GEMMs in low latency
    (300, 256, 33, 2)            generic normalize_rows_kernel with nan_empty
    (513, 1536, 1203, 2)         normalize_split_kernel<12> with nan_empty; 256-wide tiles on the negative GEMM
  Every stage case has an empty mask: its obj_feats row and its similarities must be NaN, and only they.

Measured on one B200 (1000 W power limit), largest normalised error per case (tolerance in brackets):
  fill_pool_batch sums / wsums:
    (16, 1024, 37x37)  5.5e-8 / 1.07e-7 [1.07e-5 / 2.9e-6]   (5, 1536, 37x37)    5.1e-8 / 3.8e-8 [1.07e-5 / 2.9e-6]
    (3, 1000, 37x37)   3.7e-8 / 1.4e-8  [1.07e-5 / 2.9e-6]   (3, 1022, 32x32)    6.1e-8 / 5.1e-9 [8.1e-6 / 2.2e-6]
    (2, 66, 24x40)     3.5e-8 / 2.1e-8  [7.6e-6 / 2.1e-6]    (2, 384, 74x74)     4.9e-8 / 5.5e-8 [4.1e-5 / 1.06e-5]
    (1, 64, 37x37)     2.1e-8 / 7.4e-8  [1.07e-5 / 2.9e-6]   (1, 64, 32x32)      3.5e-8 / 1.3e-8 [8.1e-6 / 2.2e-6]
    (2, 128, 112x112)  3.7e-8 / 6.2e-8  [9.4e-5 / 2.4e-5]    (1, 8, 224x224)     2.0e-8 / 9.6e-8 [3.7e-4 / 9.4e-5]
  proto_prepare: (1203, 10, 1024) 9.6e-8 [3.0e-6]   (80, 30, 1536) 1.17e-7 [5.1e-6]   (240, 1, 1024) 4.7e-8 [2.4e-6]
                 (37, 5, 100) 6.6e-8 [1.0e-6]
  bank 80 x 10 x 1024, both fill paths: sums 1.78e-7, wsums 0, prototypes 1.02e-7
  similarity_neg_top1 [TOL_SIM = 3e-5]: (1, 384, 1, 1) 5.0e-7   (128, 100, 9, 5) 1.63e-6   (129, 1024, 80, 3) 2.33e-6
                 (513, 1024, 1203, 2) 2.46e-6   (300, 1536, 80, 1) 3.15e-6   sigma 0.05: 5.5e-7   sigma 10: 3.83e-6
  stage obj / sim [5e-5 / 3e-5], ordered | unordered | low latency (ordered and unordered gave identical values):
    (129, 768, 9, 3)     1.42e-5 / 2.51e-6 | same | 1.41e-5 / 7.9e-7
    (1024, 1024, 80, 3)  1.43e-5 / 3.65e-6 | same | 1.43e-5 / 8.4e-7
    (300, 256, 33, 2)    1.04e-5 / 1.70e-6 | same | 1.04e-5 / 1.31e-6
    (513, 1536, 1203, 2) 1.54e-5 / 5.11e-6 | same | 1.54e-5 / 5.19e-6
The fill and prototype errors sit two orders of magnitude below their a-priori bounds, as expected for sums of mixed
signs; the smallest emulated defect (a dropped last patch, 7.7e-4 at 32x32) is 95x TOL_FILL.
"""
import importlib
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bank_ref import (exact_nearest_index, fill64, finalize32, nearest_index, neg64, neg_formula, neg_terms, proto64,
                      tol_fill, tol_proto, tol_wsum)
from gemm_ref import TOL_POOL, TOL_SIM, check_labels, normalised_error, pooled64, project64
from oracle import ref_torch

DEV = "cuda:0"
DEFECT_MARGIN = 4.0  # an emulated defect must exceed the tolerance by this factor
SMEM_DEFAULT = 48 * 1024  # fill_pool_kernel opts in to more dynamic shared memory above this
SMEM_LIMIT = 200 * 1024   # ... and refuses above this

FILL_CASES = [(16, 1024, (37, 37), (518, 518), "product"), (5, 1536, (37, 37), (480, 640), "nonsquare"),
              (3, 1000, (37, 37), (74, 74), "tail"), (3, 1022, (32, 32), (1000, 1000), "scalar"),
              (2, 66, (24, 40), (333, 500), "scalar_nonsquare"), (2, 384, (74, 74), (768, 768), "fp32_index"),
              (1, 64, (37, 37), (18, 18), "upscale"), (1, 64, (32, 32), (16, 16), "upscale_x2"),
              (2, 128, (112, 112), (200, 200), "smem_dynamic"), (1, 8, (224, 224), (224, 224), "smem_limit")]
PROTO_CASES = [(1203, 10, 1024), (80, 30, 1536), (240, 1, 1024), (37, 5, 100)]
NEG_CASES = [(1, 384, 1, 1, 0.8), (128, 100, 9, 5, 0.8), (129, 1024, 80, 3, 0.8), (513, 1024, 1203, 2, 0.8),
             (300, 1536, 80, 1, 0.8), (200, 768, 40, 4, 0.05), (200, 768, 40, 4, 10.0)]
STAGE_CASES = [(129, 768, 9, 3), (1024, 1024, 80, 3), (300, 256, 33, 2), (513, 1536, 1203, 2)]
STAGE_MODES = ["ordered", "unordered", "low_latency"]


def _pkg(name=""):
    return importlib.import_module("no-time-to-train_b200" + name)


def case_seed(*key) -> int:
    return 2000 + sum((i + 1) * int(round(float(np.sum(k)) * 100)) for i, k in enumerate(key)) % 100000


def _report(kind, case, **vals):
    print(f"[bank accuracy] {kind} {case} " + " ".join(f"{k} {v:.3e}" for k, v in vals.items()))


def pad64(x: int) -> int:
    return (x + 63) // 64 * 64


# ------------------------------------------------------------------------------------------------ fill inputs
def box_mask(mh, mw, gen):
    """A box with a soft rim, the recipe of synth.make_ref_shot_device on an mh x mw mask."""
    g = torch.rand(4, generator=gen).tolist()
    y0, x0 = int(g[0] * mh / 2), int(g[1] * mw / 2)
    hh, ww = int(mh / 8 + g[2] * mh * 3 / 8), int(mw / 8 + g[3] * mw * 3 / 8)
    m = torch.zeros((mh, mw))
    m[y0:y0 + hh, x0:x0 + ww] = 1.0
    rim = max(min(mh, mw) // 37, 1)
    m[y0:y0 + rim, x0:x0 + ww] = 0.5
    m[y0:y0 + hh, x0:x0 + rim] = 0.25
    return m


def fill_inputs(shots, c, grid, mask_hw, seed):
    """feat [shots, E, c] of mixed signs with a few columns scaled by 1e3 and 1e-3; soft masks [shots, mh, mw] cycling
    through full-support rand masks (non-zero everywhere), boxes with a soft rim and (from three shots on) all zeros."""
    gen = torch.Generator().manual_seed(seed)
    e = grid[0] * grid[1]
    feat = torch.randn(shots, e, c, generator=gen)
    feat[..., 0] *= 1e3
    feat[..., c // 2] *= 1e3
    feat[..., 1] *= 1e-3
    feat[..., c - 1] *= 1e-3
    kinds = ["rand", "box", "zero"] if shots >= 3 else ["rand", "box"]
    soft = torch.zeros((shots,) + tuple(mask_hw))
    for i in range(shots):
        kind = kinds[i % len(kinds)]
        if kind == "rand":
            soft[i] = 0.001 + 0.999 * torch.rand(mask_hw, generator=gen)
        elif kind == "box":
            soft[i] = box_mask(*mask_hw, gen)
    return feat.contiguous(), soft.contiguous()


def fill_smem(grid) -> int:
    e = grid[0] * grid[1]
    return 4 * (((e + 3) & ~3) + 8 * 128)


def assert_fill_branch(c, grid, mask_hw, branch):
    """The host-side geometry of fill_pool_kernel's launch (fill.cu launch_fill_pool) reaches the case's branch."""
    (eh, ew), (mh, mw) = grid, mask_hw
    e, strips, smem = eh * ew, math.ceil(c / 128), fill_smem(grid)
    assert smem <= SMEM_LIMIT
    if branch == "product":
        assert strips == 8 and c % 4 == 0 and mh == 14 * eh and mw == 14 * ew
    elif branch == "nonsquare":
        assert strips == 12 and mh != mw and mh % eh and mw % ew
    elif branch == "tail":
        assert c % 4 == 0 and c % 128 == 104 and strips == 8
    elif branch == "scalar":
        assert c % 4 != 0 and e % 8 == 0 and strips == 8
    elif branch == "scalar_nonsquare":
        assert c % 4 != 0 and e % 8 == 0 and eh != ew
    elif branch == "fp32_index":
        dst = np.arange(eh)
        diff = nearest_index(dst, mh, eh) != exact_nearest_index(dst, mh, eh)
        assert diff[37] and nearest_index(37, mh, eh) == 383
    elif branch == "upscale":
        assert mh < eh and mw < ew and eh != 2 * mh
    elif branch == "upscale_x2":
        assert eh == 2 * mh and ew == 2 * mw
    elif branch == "smem_dynamic":
        assert SMEM_DEFAULT < smem < SMEM_LIMIT
    elif branch == "smem_limit":
        assert smem == SMEM_LIMIT
    else:
        raise AssertionError(branch)


# ------------------------------------------------------------------------------------------------ CPU: references
def test_nearest_index_matches_aten():
    """nearest_index equals aten's CPU F.interpolate(mode="nearest") for every (mask, grid) size the GPU cases use,
    along each axis; at 768 -> 74 it differs from exact arithmetic (so the GPU case tells the two apart)."""
    sizes = {(m, g) for _, _, grid, mask, _ in FILL_CASES for m, g in zip(mask, grid)} | {(225, 225), (518, 37)}
    for in_size, out_size in sorted(sizes):
        x = torch.arange(in_size, dtype=torch.float64).reshape(1, 1, in_size, 1)
        want = F.interpolate(x, size=(out_size, 1), mode="nearest").flatten().to(torch.int64).numpy()
        got = nearest_index(np.arange(out_size), in_size, out_size)
        assert np.array_equal(got, want), (in_size, out_size)
    dst = np.arange(74)
    fp32, exact = nearest_index(dst, 768, 74), exact_nearest_index(dst, 768, 74)
    assert fp32[37] == 383 and exact[37] == 384
    assert np.count_nonzero(fp32 != exact) >= 1


def test_finalize32_matches_bank_postprocess():
    """finalize32 against ref_torch.bank_postprocess (the reference's formula on a raw bank) on a partly filled bank
    with one empty class, within float tolerance: the two sum in different orders."""
    gen = torch.Generator().manual_seed(17)
    n_cls, shots, e, c = 4, 3, 49, 24
    bank = ref_torch.RawBank(n_cls, shots, e, c)
    feats = torch.randn(n_cls, shots, e, c, generator=gen)
    masks = torch.rand(n_cls, shots, e, generator=gen)
    fill = [(0, 3), (1, 1), (3, 2)]  # class 2 stays empty
    for ci, k in fill:
        for _ in range(k):
            ref_torch.bank_fill(bank, [ci], feats[ci, bank.fill_counts[ci]].unsqueeze(0),
                                masks[ci, bank.fill_counts[ci]].unsqueeze(0))
    want_avg, want_ins = ref_torch.bank_postprocess(bank)
    sums = (bank.feats * bank.masks.unsqueeze(-1)).sum(dim=2)
    ins, avg = finalize32(sums, bank.masks.sum(dim=2))
    assert bool((bank.masks.sum(dim=2) == 0).any()) and bool((bank.masks[2] == 0).all())
    torch.testing.assert_close(ins, want_ins, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(avg, want_avg, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("shots,c,grid,mask_hw,branch", FILL_CASES)
def test_fill_window(shots, c, grid, mask_hw, branch):
    """On the inputs of the GPU fill cases: a correct fp32 sum of the same products in another order (torch.sum) stays
    within TOL_FILL and TOL_WSUM; dropping the last patch (E <= 1369) or one warp's partial exceeds TOL_FILL by
    DEFECT_MARGIN."""
    feat, soft = fill_inputs(shots, c, grid, mask_hw, case_seed(shots, c, grid, mask_hw))
    e = grid[0] * grid[1]
    sum64, wsum64, m, bound, wbound = fill64(feat, soft, grid)
    tol, tolw = tol_fill(e), tol_wsum(e)
    other = (m.unsqueeze(-1) * feat).sum(dim=1)
    err = normalised_error(other, sum64, bound, "fp32 sum in torch's order")
    errw = normalised_error(m.sum(dim=1), wsum64, wbound, "fp32 weight sum in torch's order")
    m64, f64 = m.to(torch.float64), feat.to(torch.float64)
    no_last = sum64 - m64[:, -1:] * f64[:, -1]
    no_warp = sum64 - torch.bmm(m64[:, 7::8].unsqueeze(1), f64[:, 7::8]).squeeze(1)
    e_last = normalised_error(no_last, sum64, bound, "no last patch")
    e_warp = normalised_error(no_warp, sum64, bound, "no warp 7")
    _report("fill window", (shots, c, grid, mask_hw), torch_order=err, tol=tol, wsum=errw, tol_wsum=tolw,
            no_last_patch=e_last, no_warp_partial=e_warp)
    assert err <= tol and errw <= tolw
    if e <= 1369:
        assert e_last >= DEFECT_MARGIN * tol
    assert e_warp >= DEFECT_MARGIN * tol


# ------------------------------------------------------------------------------------------------ neg inputs
def neg_inputs(n, c, n_cls, l_neg, seed):
    """Unit rows: obj [n, c] fp32, pos [n_cls, c] fp32, neg [n_cls * l_neg, c] fp32.  Negatives lie near their class's
    positive prototype (cosine ~0.75); objects mix their class's positive and one of its negatives (every fifth row
    is noise), so that sim_neg > sim_pos > 0 and sim_pos < 0 both occur."""
    gen = torch.Generator().manual_seed(seed)
    pos = F.normalize(torch.randn(n_cls, c, generator=gen, dtype=torch.float64), dim=-1)
    neg = F.normalize(pos.unsqueeze(1) + 0.9 * F.normalize(torch.randn(n_cls, l_neg, c, generator=gen,
                                                                       dtype=torch.float64), dim=-1), dim=-1)
    k = torch.randint(0, n_cls, (n,), generator=gen)
    li = torch.randint(0, l_neg, (n,), generator=gen)
    a, b = torch.rand(n, 1, generator=gen, dtype=torch.float64), torch.rand(n, 1, generator=gen, dtype=torch.float64)
    noise = F.normalize(torch.randn(n, c, generator=gen, dtype=torch.float64), dim=-1)
    obj = F.normalize(a * pos[k] + (0.3 + b) * neg[k, li] + 0.5 * noise, dim=-1)
    obj[4::5] = noise[4::5]
    return obj.float(), pos.float(), neg.reshape(n_cls * l_neg, c).float()


def neg_defects(obj, pos, neg, l_neg, sigma):
    """-> (sim64, bound, {defect: sim}) in float64 on the fp32 inputs."""
    sp_raw, sn_all, _, _ = neg_terms(obj, pos, neg, l_neg)
    sn = sn_all.max(dim=-1).values
    sn_but_last = sn_all[..., :-1].max(dim=-1).values if l_neg > 1 else torch.zeros_like(sn)
    ref, bound = neg64(obj, pos, neg, l_neg, sigma)
    return ref, bound, dict(max_without_last_slot=neg_formula(sp_raw, sn_but_last, sigma),
                            no_clamp_pos=neg_formula(sp_raw, sn, sigma, clamp_pos=False),
                            sigma_multiplied=neg_formula(sp_raw, sn, sigma, div_sigma=False)), sp_raw, sn


@pytest.mark.parametrize("n,c,n_cls,l_neg,sigma", NEG_CASES)
def test_neg_window(n, c, n_cls, l_neg, sigma):
    """On the inputs of the per-op negative cases, each emulated defect exceeds TOL_SIM by DEFECT_MARGIN, and the inputs
    reach both branches: a real share of elements with sim_neg > sim_pos > 0, and elements with sim_pos < 0.  (The
    1 x 1 case is a single element: its defects are only reported.)"""
    obj, pos, neg = neg_inputs(n, c, n_cls, l_neg, case_seed(n, c, n_cls, l_neg, sigma))
    ref, bound, defects, sp_raw, sn = neg_defects(obj, pos, neg, l_neg, sigma)
    errs = {k: normalised_error(v, ref, bound, k) for k, v in defects.items()}
    active = float(((sn > sp_raw) & (sp_raw > 0)).double().mean())
    _report("neg window", (n, c, n_cls, l_neg, sigma), active_share=active, **errs)
    if n * n_cls > 1:
        assert active >= 0.05 and bool((sp_raw < 0).any())
        for k, v in errs.items():
            assert v >= DEFECT_MARGIN * TOL_SIM, f"emulated defect {k}: {v:.2e} < {DEFECT_MARGIN} x {TOL_SIM:.1e}"


def stage_neg_inputs(n, c, n_cls, l_neg):
    """make_stage_inputs(degenerate=True) with l_neg + 1 bank slots per class: slot 0 is the class-level average, the
    rest are the negatives (close to it: the clustered bank), so the negative term is active."""
    inp = _pkg(".synth").make_stage_inputs(n, c, n_cls, l_neg + 1, ori_hw=(480, 640), seed=case_seed(n, c, n_cls, l_neg),
                                          e_side=37, clustered=True, degenerate=True)
    return inp, inp.feats_ins_avg[:, 0].contiguous(), inp.feats_ins_avg[:, 1:].contiguous()


def sim_splits(n, cols, c, sm_count) -> int:
    """The split-K partials of one similarity GEMM in low latency: gemm_tc_pick_splits (gemm_tc.cu) restated with the
    device's SM count, capped at kMaxSimSplits = 8, as launch_gemm_tc realises it."""
    k_blocks = 3 * pad64(c) // 64
    tiles = math.ceil(cols / 64) * math.ceil(n / 128)
    want = max(1, min(min(sm_count, 148) // tiles, 8, k_blocks))
    per = math.ceil(k_blocks / want)
    return math.ceil(k_blocks / per)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ops():
    return _pkg(".ops")


@pytest.mark.gpu
@pytest.mark.parametrize("shots,c,grid,mask_hw,branch", FILL_CASES)
def test_fill_pool_batch_per_element(ops, shots, c, grid, mask_hw, branch):
    """`ops.fill_pool_batch` against fill64: sums within TOL_FILL, weight sums within TOL_WSUM, low-res masks equal to
    the gathered soft masks.  Outputs start as NaN, so an element the kernel never writes fails."""
    assert_fill_branch(c, grid, mask_hw, branch)
    feat, soft = fill_inputs(shots, c, grid, mask_hw, case_seed(shots, c, grid, mask_hw))
    fd, sd = feat.to(DEV), soft.to(DEV)
    e = grid[0] * grid[1]
    sums = torch.full((shots, c), float("nan"), device=DEV)
    wsums = torch.full((shots,), float("nan"), device=DEV)
    lowres = torch.full((shots, e), float("nan"), device=DEV)
    ops.fill_pool_batch(fd, sd, grid, sums, wsums, lowres)
    sum64, wsum64, m, bound, wbound = fill64(fd, sd, grid)
    assert torch.equal(lowres, m), "low-res masks differ from the nearest-gathered soft masks"
    err = normalised_error(sums, sum64, bound, "sums")
    errw = normalised_error(wsums, wsum64, wbound, "wsums")
    _report("fill_pool_batch", (shots, c, grid, mask_hw), sums=err, tol=tol_fill(e), wsums=errw, tol_wsum=tol_wsum(e))
    assert err <= tol_fill(e)
    assert errw <= tol_wsum(e)


@pytest.mark.gpu
def test_fill_pool_refuses_beyond_shared_memory(ops):
    """A 225 x 225 grid needs more than 200 KB of shared memory: the call raises and writes nothing."""
    grid = (225, 225)
    assert fill_smem(grid) > SMEM_LIMIT
    feat, soft = fill_inputs(1, 8, grid, grid, 5)
    sums = torch.full((1, 8), 7.0, device=DEV)
    wsums = torch.full((1,), 7.0, device=DEV)
    lowres = torch.full((1, 225 * 225), 7.0, device=DEV)
    with pytest.raises(_pkg("._lib").NtttError):
        ops.fill_pool_batch(feat.to(DEV), soft.to(DEV), grid, sums, wsums, lowres)
    torch.cuda.synchronize()
    assert bool((sums == 7.0).all()) and bool((wsums == 7.0).all()) and bool((lowres == 7.0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("c,grid,mask_hw", [(1024, (37, 37), (518, 518)), (66, (24, 40), (333, 500))])
def test_fill_pool_accumulate_adds_the_batch_result(ops, c, grid, mask_hw):
    """`ops.fill_pool_accumulate` into a slot that holds data equals old + fill_pool_batch(the same shot), bit for bit,
    for the sums, the weight sum and the low-res mask: one fp32 add of the same fixed-order value."""
    shots = 2
    feat, soft = fill_inputs(shots, c, grid, mask_hw, case_seed(c, grid, mask_hw))
    fd, sd = feat.to(DEV), soft.to(DEV)
    e = grid[0] * grid[1]
    gen = torch.Generator().manual_seed(c)
    for i in range(shots):
        sums, wsums, lowres = (torch.empty((1, c), device=DEV), torch.empty((1,), device=DEV),
                               torch.empty((1, e), device=DEV))
        ops.fill_pool_batch(fd[i:i + 1], sd[i:i + 1], grid, sums, wsums, lowres)
        old_s = torch.randn(c, generator=gen).to(DEV)
        old_w = torch.rand(1, generator=gen).to(DEV)
        old_m = torch.rand(e, generator=gen).to(DEV)
        s, w, m = old_s.clone(), old_w.clone(), old_m.clone()
        ops.fill_pool_accumulate(fd[i], sd[i], grid, s, w, m)
        assert torch.equal(s, old_s + sums[0]), f"shot {i}: sums"
        assert torch.equal(w, old_w + wsums), f"shot {i}: weight sum"
        assert torch.equal(m, old_m + lowres[0]), f"shot {i}: low-res mask"


@pytest.mark.gpu
@pytest.mark.parametrize("with_masks", [True, False])
def test_fill_scatter_adds_rows_into_their_slots(ops, with_masks):
    """`ops.fill_scatter` with out-of-order slots and skipped rows (slot < 0) at c = 1024, e = 1369: every destination is
    before + row bit for bit, every other slot unchanged (masks given, or NULL)."""
    gen = torch.Generator().manual_seed(23)
    n, n_slots, c, e = 12, 20, 1024, 1369
    slot = torch.randperm(n_slots, generator=gen)[:n].to(torch.int32)
    slot[2] = slot[7] = -1
    sums, wsums, lowres = torch.randn(n, c, generator=gen), torch.rand(n, generator=gen), torch.rand(n, e, generator=gen)
    before = (torch.randn(n_slots, c, generator=gen), torch.randn(n_slots, generator=gen),
              torch.randn(n_slots, e, generator=gen))
    fs, ms, mk = (t.to(DEV) for t in before)
    ops.fill_scatter(sums.to(DEV), wsums.to(DEV), lowres.to(DEV), slot.to(DEV), fs, ms, mk if with_masks else None)
    want_fs, want_ms, want_mk = (t.clone() for t in before)
    live = slot >= 0
    dst = slot[live].long()
    want_fs[dst] = (before[0][dst].to(DEV) + sums[live].to(DEV)).cpu()
    want_ms[dst] = (before[1][dst].to(DEV) + wsums[live].to(DEV)).cpu()
    if with_masks:
        want_mk[dst] = (before[2][dst].to(DEV) + lowres[live].to(DEV)).cpu()
    assert torch.equal(fs.cpu(), want_fs) and torch.equal(ms.cpu(), want_ms) and torch.equal(mk.cpu(), want_mk)


def finalize_inputs(n_cls, shots, c, seed):
    """feats_sum / mask_sum of a partly filled bank: unfilled slots (zero sums, zero weight), class 5 empty, one slot
    with the tiny non-zero weight 2^-100."""
    gen = torch.Generator().manual_seed(seed)
    s = torch.randn(n_cls, shots, c, generator=gen)
    w = 1.0 + 300.0 * torch.rand(n_cls, shots, generator=gen)
    unfilled = (torch.arange(n_cls).unsqueeze(1) + torch.arange(shots).unsqueeze(0)) % 7 == 3
    s[unfilled] = 0.0
    w[unfilled] = 0.0
    s[5], w[5] = 0.0, 0.0
    w[7, 2] = 2.0 ** -100
    return s, w


@pytest.mark.gpu
def test_fill_finalize_bit_exact(ops):
    """`ops.fill_finalize` at 1203 classes x 10 shots x 1024 equals finalize32 of its own inputs bit for bit."""
    s, w = finalize_inputs(1203, 10, 1024, 29)
    assert bool((w == 0).any()) and float(w[5].sum()) == 0.0 and 0.0 < float(w[7, 2]) < 1e-30
    ins, avg = ops.fill_finalize(s.to(DEV), w.to(DEV))
    want_ins, want_avg = finalize32(s, w)
    assert torch.equal(ins.cpu(), want_ins), "feats_ins_avg differs from finalize32"
    assert torch.equal(avg.cpu(), want_avg), "feats_avg differs from finalize32"


def proto_inputs(n_cls, shots, c, seed):
    """Bank slots near five cluster centres, every seventh slot unfilled (zeros, when shots > 1), class 3 all zeros."""
    gen = torch.Generator().manual_seed(seed)
    centres = F.normalize(torch.randn(5, c, generator=gen), dim=-1)
    x = centres[torch.arange(n_cls) % 5].unsqueeze(1) + (1.0 / math.sqrt(c)) * torch.randn(n_cls, shots, c, generator=gen)
    if shots > 1:
        x[((torch.arange(n_cls).unsqueeze(1) + torch.arange(shots).unsqueeze(0)) % 7 == 3)] = 0.0
    x[3] = 0.0
    return x.contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("n_cls,shots,c", PROTO_CASES)
def test_proto_prepare_per_element(ops, n_cls, shots, c):
    """`ops.proto_prepare` against proto64 of its own input; the zero class row comes out as exact zeros."""
    x = proto_inputs(n_cls, shots, c, case_seed(n_cls, shots, c)).to(DEV)
    got = ops.proto_prepare(x)
    want, bound = proto64(x)
    assert bool((bound[3] == 0).all())
    err = normalised_error(got, want, bound, "proto")
    _report("proto_prepare", (n_cls, shots, c), proto=err, tol=tol_proto(shots, c))
    assert err <= tol_proto(shots, c)


@pytest.mark.gpu
def test_bank_to_prototypes_at_the_product_shape(pkg):
    """An 80-class x 10-slot bank at c = 1024, E = 1369 from 518 x 518 soft masks, some slots unfilled and class 7 empty,
    filled shot by shot (MemoryBank.fill: the accumulate path) and in batches of 16 (fill_batch: pool + scatter).  The
    two banks are bit-identical, and each passes the fill, finalize and prototype checks on its own intermediates."""
    n_cls, length, grid, c = 80, 10, (37, 37), 1024
    e = grid[0] * grid[1]
    synth = pkg.synth
    centres = synth.cluster_centres(c)
    counts = [0 if k == 7 else length - k % 3 for k in range(n_cls)]  # 712 shots: 44 full batches of 16 and one of 8
    order = [(k, r) for r in range(length) for k in range(n_cls) if r < counts[k]]
    cfg = {"category_num": n_cls, "length": length, "feat_shape": (e, c)}
    one, batched = pkg.MemoryBank(cfg).to(DEV), pkg.MemoryBank(cfg).to(DEV)
    sum64 = torch.zeros((n_cls, length, c), dtype=torch.float64, device=DEV)
    bound = torch.zeros_like(sum64)
    wsum64 = torch.zeros((n_cls, length), dtype=torch.float64, device=DEV)
    wbound = torch.zeros_like(wsum64)
    lowres = torch.zeros((n_cls, length, e), device=DEV)
    for i0 in range(0, len(order), 16):
        chunk = order[i0:i0 + 16]
        shots = [synth.make_ref_shot_device(k, r, centres, DEV) for k, r in chunk]
        feats = torch.stack([f for f, _ in shots])
        masks = torch.stack([m for _, m in shots])
        for (k, _), (f, m) in zip(chunk, shots):
            one.fill(k, f, m, grid)
        batched.fill_batch([k for k, _ in chunk], feats, masks, grid)
        s, w, lr, b, wb = fill64(feats, masks, grid)
        for j, (k, r) in enumerate(chunk):
            sum64[k, r] += s[j]
            bound[k, r] += b[j]
            wsum64[k, r] += w[j]
            wbound[k, r] += wb[j]
            lowres[k, r] += lr[j]
    for name in ("feats_sum", "mask_sum", "masks", "fill_counts"):
        assert torch.equal(getattr(one, name), getattr(batched, name)), f"{name}: the two fill paths differ"
    assert one.fill_counts.tolist() == counts
    stage = pkg.MatchingStage(DEV, pkg.StageConfig(enc_hw=grid))
    for label, bank in (("one by one", one), ("batched", batched)):
        assert torch.equal(bank.masks, lowres), f"{label}: low-res masks"
        err = normalised_error(bank.feats_sum, sum64, bound, f"{label}: feats_sum")
        errw = normalised_error(bank.mask_sum, wsum64, wbound, f"{label}: mask_sum")
        fs, ms = bank.feats_sum.cpu(), bank.mask_sum.cpu()
        bank.postprocess()
        want_ins, want_avg = finalize32(fs, ms)
        assert torch.equal(bank.feats_ins_avg.cpu(), want_ins), f"{label}: feats_ins_avg differs from finalize32"
        assert torch.equal(bank.feats_avg.cpu(), want_avg), f"{label}: feats_avg differs from finalize32"
        stage.set_prototypes(bank.feats_ins_avg)
        want_p, bound_p = proto64(bank.feats_ins_avg)
        assert bool((bound_p[7] == 0).all())
        err_p = normalised_error(stage.proto, want_p, bound_p, f"{label}: prototypes")
        _report("bank", label, sums=err, tol=tol_fill(e), wsums=errw, tol_wsum=tol_wsum(e), proto=err_p,
                tol_proto=tol_proto(length, c))
        assert err <= tol_fill(e) and errw <= tol_wsum(e) and err_p <= tol_proto(length, c)


@pytest.mark.gpu
@pytest.mark.parametrize("n,c,n_cls,l_neg,sigma", NEG_CASES)
def test_similarity_neg_top1_per_element(ops, n, c, n_cls, l_neg, sigma):
    """`ops.similarity_neg_top1` against neg64 of the same fp32 rows; labels are the kernel's own argmax and the float64
    argmax outside the band; the top score is sim[label] (with the k == n_cls rule for one class)."""
    cols = n_cls * l_neg
    if n_cls == 1:
        assert n == 1 and l_neg == 1
    if c == 100:
        assert c % 64 != 0 and pad64(c) == 128
    if cols == 240:
        assert n_cls == 80 and l_neg == 3
    if n_cls == 1203:  # 256-wide tiles (launch_gemm_tc: N, M >= 512 outside low latency), N tails on both products
        assert n >= 512 and n_cls >= 512 and cols >= 512 and n_cls % 256 and cols % 256
    obj, pos, neg = neg_inputs(n, c, n_cls, l_neg, case_seed(n, c, n_cls, l_neg, sigma))
    od = obj.to(DEV)
    sim, top_score, top_label = ops.similarity_neg_top1(od, pos.to(DEV), neg.to(DEV), l_neg, sigma)
    ref, bound = neg64(od, pos.to(DEV), neg.to(DEV), l_neg, sigma)
    if sigma != 0.8:  # steep / flat decay: the decay must actually act
        sp_raw, sn_all, _, _ = neg_terms(od, pos.to(DEV), neg.to(DEV), l_neg)
        assert bool(((sn_all.max(-1).values > sp_raw) & (sp_raw > 0)).any())
    err = normalised_error(sim, ref, bound, "sim")
    flips = check_labels(sim, ref, bound, "sim", labels=top_label)
    best = sim.gather(1, top_label.long().unsqueeze(1)).squeeze(1)
    if n_cls == 1:
        best = best * (best > best * 0.6)
    assert torch.equal(top_score, best)
    _report("similarity_neg_top1", (n, c, n_cls, l_neg, sigma), sim=err, tol=TOL_SIM, label_flips=flips)
    assert err <= TOL_SIM


_stage_refs = {}


def _stage_case(pkg, n, c, n_cls, l_neg):
    """Inputs, the stage with negative prototypes and the float64 pooled reference (cached: each case runs in three
    modes)."""
    key = (n, c, n_cls, l_neg)
    if key not in _stage_refs:
        _stage_refs.clear()
        inp, pos, neg = stage_neg_inputs(n, c, n_cls, l_neg)
        stage = pkg.MatchingStage(DEV, pkg.StageConfig(nms_thr=0.5, num_out_instance=20, enc_hw=(37, 37)))
        stage.set_prototypes_with_negatives(pos, neg)
        d = inp.lr_masks.to(DEV)
        area = ref_torch.threshold_lowres(d).sum(1)
        feat = inp.tar_feat.to(DEV)
        obj64, bound = pooled64(project64(d, (37, 37)), feat.double(), area)
        pos64 = F.normalize(pos.double(), dim=-1).to(DEV)
        neg64_ = F.normalize(neg.double(), dim=-1).reshape(n_cls * l_neg, c).to(DEV)
        _stage_refs[key] = (stage, (d, inp.pred_ious.to(DEV), feat, inp.ori_hw), area, obj64, bound, pos64, neg64_)
    return _stage_refs[key]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", STAGE_MODES)
@pytest.mark.parametrize("n,c,n_cls,l_neg", STAGE_CASES)
def test_stage_with_negatives_per_element(pkg, n, c, n_cls, l_neg, mode):
    """`set_prototypes_with_negatives` + `match(taps=True)`: obj_feats NaN exactly on the empty-mask rows and within
    TOL_POOL of the float64 pooled rows elsewhere; sim all NaN on the empty-mask rows and within TOL_SIM of neg64 of the
    kernel's own obj_feats elsewhere; labels as in the per-op test."""
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    cols = n_cls * l_neg
    if (n, c) == (129, 768):  # low latency splits both similarity GEMMs
        assert sim_splits(n, n_cls, c, sm) > 1 and sim_splits(n, cols, c, sm) > 1
    if (n, c) == (1024, 1024):  # ordered pooling (api.cu nttt_match_image: n > 128, <= 32 k-blocks, vector width)
        assert 128 < n <= 8192 and pad64(37 * 37) // 64 <= 32 and c in (384, 768, 1024, 1536)
    if c == 256:  # no normalize_split_kernel instance: the generic normalize_rows_kernel runs
        assert c % 128 == 0 and c // 128 not in (3, 6, 8, 12)
    if c == 1536:  # normalize_split_kernel<12>; 256-wide tiles on the negative GEMM outside low latency
        assert c // 128 == 12 and n >= 512 and cols >= 512
    stage, args, area, obj64, bound_obj, pos64, neg64_ = _stage_case(pkg, n, c, n_cls, l_neg)
    try:
        stage.tune("pool_order", 0 if mode == "unordered" else 1)
        out = stage.match(*args, taps=True, low_latency=mode == "low_latency")
    finally:
        stage.tune("pool_order", 1)
    obj, sim = out["taps"]["obj_feats"], out["taps"]["sim"]
    empty = area == 0
    assert bool(empty.any()), "the case has no empty mask"
    assert bool(torch.isnan(obj[empty]).all()) and bool(torch.isnan(sim[empty]).all())
    live = ~empty
    err_obj = normalised_error(obj[live], obj64[live], bound_obj[live], "obj_feats")
    ref, bound = neg64(obj[live], pos64, neg64_, l_neg, stage.cfg.neg_sigma)
    err_sim = normalised_error(sim[live], ref, bound, "sim")
    flips = check_labels(sim[live], ref, bound, "sim")
    _report("stage neg", (n, c, n_cls, l_neg, mode), obj=err_obj, tol_obj=TOL_POOL, sim=err_sim, tol_sim=TOL_SIM,
            label_flips=flips)
    assert err_obj <= TOL_POOL
    assert err_sim <= TOL_SIM
