"""Accuracy of the split-bf16 tensor-core contractions against float64 references, per element.

Both float contractions of the stage run on the tcgen05 GEMM of csrc/gemm_tc.cu: the pooling product
`sums = proj . feat` and the similarity product `sim = obj_feats . proto^T`.  Each fp32 operand x is split into
hi = bf16(x), lo = bf16(x - hi), and A' = [hi | hi | lo], B' = [hi | lo | hi] along K give hi.hi + hi.lo + lo.hi: the
dropped lo.lo term leaves ~2^-17 of |A|.|B|.  The golden comparisons (1e-3 of the matrix maximum) cannot tell this
scheme from one that lost a cross term; these tests can.

Metric.  For a raw product D = A B^T an element's error is |got - ref| / (|A| |B|^T), the bound that scales with the
element, not with the largest element of the matrix.  A pooled row is normalised, so its error is divided by
(|proj| |feat|) / area / ||(proj feat) / area|| (the area cancels).  Rows whose reference is exactly zero (empty masks,
the F.normalize eps clamp) must come out exactly zero.  Each GEMM is checked on its own inputs: the similarity
reference is the float64 product of the kernel's OWN obj_feats with float64 prototypes, so a pooling error can neither
hide nor inflate a similarity error.  Top-1 labels are the argmax of the kernel's own sim and agree with the float64
argmax except where the float64 top-2 gap lies inside the row's tolerance band.

The tolerances (TOL_POOL, TOL_SIM) sit at >= 2x the largest error measured on a B200 and >= 4x below the smallest
error of an emulated defect (test_emulated_*_defects_exceed_tolerance: a float64 emulation of the split scheme with
bf16 rounding that drops hi.lo, lo.hi or both, on the inputs of the GPU cases).

Measured on one B200 (1000 W power limit), max normalised error per case:
  pool_normalize obj:   (1, 37x37, 64) 5.0e-6   (127, 37x37, 66) 1.09e-5   (129, 32x32, 100) 1.24e-5
                        (513, 37x37, 768) 1.25e-5   (600, 37x37, 1000) 1.31e-5   (1000, 64x64, 1024) 9.0e-6
                        (300, 24x40, 1536) 1.60e-5
  similarity_top1 sim:  (1, 384, 1) 8.1e-8   (127, 384, 9) 1.41e-6   (128, 100, 64) 2.97e-6   (129, 1024, 65) 1.33e-6
                        (200, 768, 128) 1.44e-6   (200, 768, 129) non-negative 7.6e-6   (513, 1024, 512) 1.83e-6
                        (1000, 1024, 1203) 2.02e-6   (300, 1536, 80) 1.61e-6
  stage obj / sim, ordered | unordered | low latency (ordered and unordered gave identical values):
                        (1024, 1024, 80, 37)   1.53e-5 / 6.95e-6 | same | 1.53e-5 / 1.42e-6
                        (513, 1536, 1203, 37)  1.38e-5 / 1.01e-5 | same | 1.37e-5 / 1.02e-5
                        (129, 768, 9, 37)      1.57e-5 / 4.82e-6 | same | 1.57e-5 / 9.5e-7
                        (300, 256, 33, 37)     1.20e-5 / 3.05e-6 | same | 1.20e-5 / 2.18e-6
                        (400, 384, 80, 32)     1.16e-5 / 3.69e-6 | same | 1.16e-5 / 1.57e-6
                        (400, 384, 80, 64)     6.9e-6 / 3.62e-6  | same | 6.9e-6 / 1.67e-6
  project_masks, ulps of the row maximum against the float64 projection with the reference's float32 weights:
                        0 (bit-exact) at every power-of-two mask size; 1.6 at 96 x 160.  PROJ_ULPS = 8.
The pooled rows match the float64 emulation of the split scheme (<= 1.6e-5, dominated by the dropped lo.lo term coupled
through the row normalisation).  The stage's similarities on clustered features (cosines ~0.5-0.9) carry a further
~1e-5 that the emulation, which sums in float64, does not have: the fp32 accumulation of K' = 3 * 1024 or 3 * 1536
products in one TMEM accumulator.  The low-latency similarity split-K (up to 8 partial accumulators, added in fp32)
brings it down to the emulated level; at 1203 classes the 95 output tiles fill the machine and it does not split.  Largest: pool 1.60e-5, sim 1.02e-5; TOL_POOL = 5e-5 and TOL_SIM = 3e-5.  The smallest
emulated defects are 1.0e-3 (pool, one mask) and 2.5e-4 (sim, stage case (129, 768, 9)), 20x and 8x the tolerances.

Per-op cases and the branch each one reaches (gemm_tc.cu launch_gemm_tc, score.cu launch_normalize_split):
  pool_normalize (never split-K, never skipping, generic normalisation always), (n, grid, c):
    (1, 37x37, 64)         BN64 tile of 128 rows holding one mask
    (127, 37x37, 66)       BN128 (65..128 columns); ldd % 4 != 0 -> scalar epilogue
    (129, 32x32, 100)      K = 1024 without padding; two M tiles, the second holding one row
    (513, 37x37, 768)      BN256 (N, M >= 512), N exactly three tiles
    (600, 37x37, 1000)     BN256 with an N tail of 232
    (1000, 64x64, 1024)    64 k-blocks per K segment
    (300, 24x40, 1536)     non-square grid, E = 960 padded to 1024; BN128 (N >= 512, M < 512)
  similarity_top1 (throughput launch: never split-K), (n, c, n_cls):
    (1, 384, 1)            the reference's k == n_cls branch of the top-1 score
    (127, 384, 9), (128, 100, 64)       BN64, c = 100 padded to 128
    (129, 1024, 65), (200, 768, 128)    BN128
    (200, 768, 129)        BN64, three N tiles, tail of one column; non-negative operands
    (513, 1024, 512)       BN256
    (1000, 1024, 1203)     BN256, N tail of 179, odd ldd -> scalar epilogue
    (300, 1536, 80)        BN128 at the widest supported encoder width
  project_masks: grids 37x37, 32x32, 24x40, 64x64 on 256x256 masks, 16x16 on 128x128 masks (the coarsest grid the
    scatter tables allow) and 37x37 on 96x160 masks, degenerate masks included.

Whole-stage cases (MatchingStage.match(taps=True)), each in throughput mode with pool_order 1 and 0 and in low-latency
mode, (n, c, n_cls, grid):
    (1024, 1024, 80, 37)   ordered pooling with k-block skipping (pool_order 1); BN256 pooling; split-K 2 pooling and
                           split-K similarity in low latency; side-stream p_split; normalize_split_kernel<8>
    (513, 1536, 1203, 37)  BN256 on both GEMMs in throughput mode; ordered skipping GEMM and normalize_split_kernel<12>
                           at c = 1536
    (129, 768, 9, 37)      low latency: similarity split-K of 36 k-blocks into 8 splits, seven of 5 and one of 1
    (300, 256, 33, 37)     generic normalisation (c = 256 has no vector kernel): a_ready = false
    (400, 384, 80, 32)     K without padding, ordered at c = 384 (normalize_split_kernel<3>)
    (400, 384, 80, 64)     64 k-blocks per segment: never ordered
project_masks_kernel<true> writes the split A operand in every case, with perm / active when ordered.
"""
import importlib

import pytest
import torch
import torch.nn.functional as F

from gemm_ref import TOL_POOL, TOL_SIM, check_labels, normalised_error, pooled64, project64
from oracle import ref_torch

DEV = "cuda:0"

DEFECT_MARGIN = 4.0  # an emulated defect must exceed the tolerance by this factor
PROJ_ULPS = 8        # project_masks: fp32 accumulation within this many ulps of the row maximum

POOL_CASES = [(1, (37, 37), 64), (127, (37, 37), 66), (129, (32, 32), 100), (513, (37, 37), 768),
              (600, (37, 37), 1000), (1000, (64, 64), 1024), (300, (24, 40), 1536)]
SIM_CASES = [(1, 384, 1, False), (127, 384, 9, False), (128, 100, 64, False), (129, 1024, 65, False),
             (200, 768, 128, False), (200, 768, 129, True), (513, 1024, 512, False), (1000, 1024, 1203, False),
             (300, 1536, 80, False)]
PROJ_CASES = [((37, 37), (256, 256)), ((32, 32), (256, 256)), ((24, 40), (256, 256)), ((64, 64), (256, 256)),
              ((16, 16), (128, 128)), ((37, 37), (96, 160))]
STAGE_CASES = [(1024, 1024, 80, 37), (513, 1536, 1203, 37), (129, 768, 9, 37), (300, 256, 33, 37),
               (400, 384, 80, 32), (400, 384, 80, 64)]
STAGE_MODES = ["ordered", "unordered", "low_latency"]


def _synth():
    return importlib.import_module("no-time-to-train_b200.synth")


# ------------------------------------------------------------------------------------------------ inputs
def pool_inputs(n, enc_hw, c, seed):
    """Masks (degenerate cases included when n >= 8) and clustered target features for a pooling case."""
    synth = _synth()
    gen = torch.Generator().manual_seed(seed)
    masks = synth.make_masks(n, gen)
    if n >= 8:
        synth.inject_degenerate_cases(masks, torch.zeros(2, 2, 4))
    feat, _ = synth.make_features(enc_hw[0] * enc_hw[1], c, 4, 1, gen, clustered=True)
    return masks, feat


def sim_inputs(n, c, n_cls, nonneg, seed):
    """Unit rows: obj_feats [n, c] and prototypes [n_cls, c] (non-negative entries when `nonneg`)."""
    gen = torch.Generator().manual_seed(seed)
    obj = torch.randn(n, c, generator=gen)
    proto = torch.randn(n_cls, c, generator=gen, dtype=torch.float64)
    if nonneg:
        obj, proto = obj.abs(), proto.abs()
    return F.normalize(obj, dim=-1), F.normalize(proto, dim=-1)


def case_seed(*key) -> int:
    return 1000 + sum((i + 1) * (k if isinstance(k, int) else sum(k)) for i, k in enumerate(key)) % 100000


# ------------------------------------------------------------------------------------------------ emulation (CPU)
def split_bf16(x: torch.Tensor):
    """fp32 x -> (hi, lo) in float64, hi = bf16(x), lo = bf16(x - hi) with round-to-nearest-even, as the kernels do."""
    x = x.to(torch.float32)
    hi = x.to(torch.bfloat16)
    lo = (x - hi.to(torch.float32)).to(torch.bfloat16)
    return hi.to(torch.float64), lo.to(torch.float64)


def emulate_products(a: torch.Tensor, b: torch.Tensor):
    """The three partial products of the split scheme for D = A B^T (A [M, K], B [N, K] fp32), summed in float64:
    -> dict hh, hl (A_hi B_lo^T), lh (A_lo B_hi^T)."""
    ah, al = split_bf16(a)
    bh, bl = split_bf16(b)
    return dict(hh=ah @ bh.t(), hl=ah @ bl.t(), lh=al @ bh.t())


def emulated(parts, terms):
    out = parts["hh"].clone()
    for t in terms:
        out += parts[t]
    return out


VARIANTS = {"full": ("hl", "lh"), "no_hl": ("lh",), "no_lh": ("hl",), "plain_bf16": ()}


def emulated_pool_errors(masks, feat, enc_hw):
    """Normalised pooled-row error of each emulated variant against the float64 reference (fp32 proj and feat)."""
    proj64 = project64(masks, enc_hw)
    area = ref_torch.threshold_lowres(masks).sum(1)
    feat64 = feat.to(torch.float64)
    ref, bound = pooled64(proj64, feat64, area)
    parts = emulate_products(proj64.to(torch.float32), feat.t().contiguous())
    a = area.to(torch.float64).clamp(min=1.0).unsqueeze(1)
    out = {}
    for name, terms in VARIANTS.items():
        sums = emulated(parts, terms).to(torch.float32).to(torch.float64)
        obj = F.normalize(sums / a, dim=-1).to(torch.float32)
        out[name] = normalised_error(obj, ref, bound, f"emulated pool {name}")
    return out


def emulated_sim_errors(obj, proto64):
    proto = proto64.to(torch.float32)
    obj64 = obj.to(torch.float64)
    ref = obj64 @ proto64.t()
    bound = obj64.abs() @ proto64.abs().t()
    parts = emulate_products(obj, proto)
    return {name: normalised_error(emulated(parts, terms).to(torch.float32), ref, bound, f"emulated sim {name}")
            for name, terms in VARIANTS.items()}


def _assert_window(errs, tol, what, defects=True):
    assert errs["full"] < tol, f"{what}: the correct split scheme emulates to {errs['full']:.2e} >= {tol:.1e}"
    for name in ("no_hl", "no_lh", "plain_bf16") if defects else ():
        assert errs[name] >= DEFECT_MARGIN * tol, \
            f"{what}: emulated defect {name} gives only {errs[name]:.2e} < {DEFECT_MARGIN} x {tol:.1e}"


def test_separable_projection_matches_dense_upsample():
    """project64's separable Uy^T M Ux equals masks @ the reference's dense upsample_features(eye(E)) on a small
    non-square case: 37 -> 96 rows (a non-dyadic scale), 40 -> 128 columns."""
    enc_hw, hw = (37, 40), (96, 128)
    synth = _synth()
    masks = synth.make_masks(12, torch.Generator().manual_seed(3))
    synth.inject_degenerate_cases(masks, torch.zeros(2, 2, 4))
    masks = masks[:, :hw[0], :hw[1]].contiguous()
    dense = ref_torch.upsample_features(torch.eye(enc_hw[0] * enc_hw[1], dtype=torch.float64), enc_hw, hw)  # [P, E]
    want = ref_torch.threshold_lowres(masks).to(torch.float64) @ dense
    got = project64(masks, enc_hw, chunk=5, weights=torch.float64)
    assert float((got - want).abs().max()) <= 1e-12 * float(want.abs().max())
    # the reference's float32 weights: within a few float32 ulps of the exact ones (37 -> 96 is not dyadic)
    got32 = project64(masks, enc_hw, chunk=5)
    assert float((got32 - want).abs().max()) <= 1e-5 * float(want.abs().max())
    assert float(got[0].abs().max()) == 0.0 and float(got[1].abs().max()) > 0.0


@pytest.mark.parametrize("n,enc_hw,c", POOL_CASES)
def test_emulated_pool_defects_exceed_tolerance(n, enc_hw, c):
    """On the inputs of the per-op pooling cases, the emulated 3-term split stays below TOL_POOL and each emulated
    defect (no hi.lo, no lo.hi, plain bf16) exceeds it by DEFECT_MARGIN."""
    masks, feat = pool_inputs(n, enc_hw, c, case_seed(n, enc_hw, c))
    errs = emulated_pool_errors(masks, feat, enc_hw)
    print(f"[emulated pool n={n} grid={enc_hw} c={c}] " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    _assert_window(errs, TOL_POOL, f"pool {n}x{enc_hw}x{c}")


@pytest.mark.parametrize("n,c,n_cls,nonneg", SIM_CASES)
def test_emulated_sim_defects_exceed_tolerance(n, c, n_cls, nonneg):
    """On the inputs of the per-op similarity cases, the emulated 3-term split stays below TOL_SIM and each emulated
    defect exceeds it by DEFECT_MARGIN.  (The 1 x 1 case is a single dot product: one element is too few to expose a
    dropped term reliably, so its defects are only reported.)"""
    obj, proto64 = sim_inputs(n, c, n_cls, nonneg, case_seed(n, c, n_cls))
    errs = emulated_sim_errors(obj, proto64)
    print(f"[emulated sim n={n} c={c} n_cls={n_cls} nonneg={nonneg}] " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    _assert_window(errs, TOL_SIM, f"sim {n}x{c}x{n_cls}", defects=n * n_cls > 1)


def stage_inputs(n, c, n_cls, grid):
    return _synth().make_stage_inputs(n, c, n_cls, 2, ori_hw=(480, 640), seed=case_seed(n, c, n_cls, grid), e_side=grid,
                                      clustered=True, degenerate=True)


@pytest.mark.parametrize("n,c,n_cls,grid", STAGE_CASES)
def test_emulated_stage_defects_exceed_tolerance(n, c, n_cls, grid):
    """The same window on the inputs of the whole-stage cases: the pooling product of the masks' projection with the
    target features, then the similarity product of the (emulated, correct) pooled rows with the prototypes."""
    inp = stage_inputs(n, c, n_cls, grid)
    pool = emulated_pool_errors(inp.lr_masks, inp.tar_feat, (grid, grid))
    proj64 = project64(inp.lr_masks, (grid, grid))
    obj64, _ = pooled64(proj64, inp.tar_feat.to(torch.float64), ref_torch.threshold_lowres(inp.lr_masks).sum(1))
    sim = emulated_sim_errors(obj64.to(torch.float32), ref_torch.prototypes(inp.feats_ins_avg.to(torch.float64)))
    for kind, errs in (("pool", pool), ("sim", sim)):
        print(f"[emulated stage {kind} n={n} c={c} n_cls={n_cls} grid={grid}] " +
              " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    _assert_window(pool, TOL_POOL, f"stage pool {n}x{c}x{grid}")
    _assert_window(sim, TOL_SIM, f"stage sim {n}x{c}x{n_cls}")


# ------------------------------------------------------------------------------------------------ GPU: per op
@pytest.fixture(scope="module")
def ops():
    return importlib.import_module("no-time-to-train_b200.ops")


def _report(kind, case, **errs):
    print(f"[gemm accuracy] {kind} {case} " + " ".join(f"{k} {v:.3e}" for k, v in errs.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("enc_hw,hw", PROJ_CASES)
def test_project_masks_matches_float64(ops, enc_hw, hw):
    """`ops.project_masks` (fp32 accumulation of the antialias weights over the mask's set pixels) against proj64,
    within PROJ_ULPS ulps of each row's maximum; empty rows exactly zero.  The reference is built from the reference's
    own float32 weights, so what is measured is the kernel's fp32 accumulation.  From a power-of-two mask size every
    weight and every partial sum is dyadic and exact in fp32; 96 x 160 masks have weights that are not.  (Against the
    weights of exact arithmetic, the 96 x 160 case differs by ~30 ulps of the row maximum: the reference's own
    float32 weight rounding, which the kernel's tables reproduce on purpose.)"""
    synth = _synth()
    masks = synth.make_masks(64, torch.Generator().manual_seed(case_seed(enc_hw, hw)))
    synth.inject_degenerate_cases(masks, torch.zeros(2, 2, 4))
    oy, ox = (256 - hw[0]) // 2, (256 - hw[1]) // 2  # centre crop: the single-pixel and the line mask survive
    d = masks[:, oy:oy + hw[0], ox:ox + hw[1]].contiguous().to(DEV)
    bits, area, box, *_ = ops.threshold_pack(d)
    proj = ops.project_masks(bits, box, hw, enc_hw)
    want = project64(d, enc_hw)
    rowmax = want.abs().max(dim=1).values
    live = rowmax > 0
    assert bool((~live).any()) and bool((area[~live] == 0).all())  # the empty masks, and only they
    assert bool((proj[~live] == 0).all())
    ulp = torch.exp2(torch.floor(torch.log2(rowmax[live])) - 23)
    ulps = float(((proj[live].double() - want[live]).abs().max(dim=1).values / ulp).max())
    _report("project_masks", (enc_hw, hw), ulps_of_row_max=ulps)
    assert ulps <= PROJ_ULPS


@pytest.mark.gpu
@pytest.mark.parametrize("n,enc_hw,c", POOL_CASES)
def test_pool_normalize_per_element(ops, n, enc_hw, c):
    """`ops.pool_normalize` on the kernel's own projection, against the float64 pooled rows."""
    masks, feat = pool_inputs(n, enc_hw, c, case_seed(n, enc_hw, c))
    bits, area, box, *_ = ops.threshold_pack(masks.to(DEV))
    proj = ops.project_masks(bits, box, (256, 256), enc_hw)
    fd = feat.to(DEV)
    obj = ops.pool_normalize(proj, fd, area)
    ref, bound = pooled64(proj.double(), fd.double(), area)
    if n >= 8:
        assert bool((area == 0).any())  # an empty mask: its row must come out exactly zero
    err = normalised_error(obj, ref, bound, "obj_feats")
    _report("pool_normalize", (n, enc_hw, c), obj=err)
    assert err <= TOL_POOL


@pytest.mark.gpu
@pytest.mark.parametrize("n,c,n_cls,nonneg", SIM_CASES)
def test_similarity_top1_per_element(ops, n, c, n_cls, nonneg):
    """`ops.similarity_top1` against the float64 product of the same unit rows; top-1 labels and scores."""
    obj, proto64 = sim_inputs(n, c, n_cls, nonneg, case_seed(n, c, n_cls))
    od = obj.to(DEV)
    p64 = proto64.to(DEV)
    sim, top_score, top_label = ops.similarity_top1(od, p64.float())
    ref = od.double() @ p64.t()
    bound = od.double().abs() @ p64.abs().t()
    err = normalised_error(sim, ref, bound, "sim")
    flips = check_labels(sim, ref, bound, "sim", labels=top_label)
    best = sim.gather(1, top_label.long().unsqueeze(1)).squeeze(1)
    if n_cls == 1:
        best = best * (best > best * 0.6)  # the reference's k == n_cls branch
    assert torch.equal(top_score, best)
    _report("similarity_top1", (n, c, n_cls, "nonneg" if nonneg else "signed"), sim=err, label_flips=flips)
    assert err <= TOL_SIM


# ------------------------------------------------------------------------------------------------ GPU: whole stage
_stage_refs = {}


def _stage_case(P, n, c, n_cls, grid):
    """Inputs, the stage (prototypes set) and the float64 pooled reference of one whole-stage case (cached: every case
    runs in three modes)."""
    key = (n, c, n_cls, grid)
    if key not in _stage_refs:
        _stage_refs.clear()
        inp = stage_inputs(n, c, n_cls, grid)
        stage = P.MatchingStage(DEV, P.StageConfig(nms_thr=0.5, num_out_instance=20, enc_hw=(grid, grid)))
        stage.set_prototypes(inp.feats_ins_avg)
        d = inp.lr_masks.to(DEV)
        area = ref_torch.threshold_lowres(d).sum(1)
        feat = inp.tar_feat.to(DEV)
        obj64, bound = pooled64(project64(d, (grid, grid)), feat.double(), area)
        proto64 = ref_torch.prototypes(inp.feats_ins_avg.double()).to(DEV)
        _stage_refs[key] = (stage, (d, inp.pred_ious.to(DEV), feat, inp.ori_hw), obj64, bound, proto64)
    return _stage_refs[key]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", STAGE_MODES)
@pytest.mark.parametrize("n,c,n_cls,grid", STAGE_CASES)
def test_stage_contractions_per_element(n, c, n_cls, grid, mode):
    """`MatchingStage.match(taps=True)`: the obj_feats tap against the float64 pooled rows of the float64 projection,
    the sim tap against the float64 product of that obj_feats tap with the float64 prototypes, labels against both."""
    P = importlib.import_module("no-time-to-train_b200")
    stage, args, obj64, bound_obj, proto64 = _stage_case(P, n, c, n_cls, grid)
    try:
        stage.tune("pool_order", 0 if mode == "unordered" else 1)
        out = stage.match(*args, taps=True, low_latency=mode == "low_latency")
    finally:
        stage.tune("pool_order", 1)
    obj, sim = out["taps"]["obj_feats"], out["taps"]["sim"]
    err_obj = normalised_error(obj, obj64, bound_obj, "obj_feats")
    o64 = obj.double()
    ref = o64 @ proto64.t()
    bound = o64.abs() @ proto64.abs().t()
    err_sim = normalised_error(sim, ref, bound, "sim")
    flips = check_labels(sim, ref, bound, "sim")
    _report("stage", (n, c, n_cls, grid, mode), obj=err_obj, sim=err_sim, label_flips=flips)
    assert err_obj <= TOL_POOL
    assert err_sim <= TOL_SIM
