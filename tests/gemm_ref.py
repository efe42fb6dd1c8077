"""Float64 references and metrics of the split-bf16 contractions, shared by the accuracy tests.  The module docstring of
test_gemm_accuracy.py defines the metric and says how the tolerances were set."""
import torch
import torch.nn.functional as F

from oracle import ref_torch

# normalised error limits of the pooled rows and of the similarities (test_gemm_accuracy.py's module docstring)
TOL_POOL = 5e-5
TOL_SIM = 3e-5


def axis_weights(n_in: int, n_out: int, device="cpu", dtype=torch.float32) -> torch.Tensor:
    """U [n_out, n_in], returned as float64: the 1-D antialiased bilinear resize (align_corners=False) of n_in samples to
    n_out, read off by resizing identity rows along one axis with aten's CPU kernel.  A one-hot row resizes to exactly
    its weights, so dtype=float32 gives the weights the reference computes for its float32 features (its fp32 recipe
    of centre, support and normalisation), which the product's tables reproduce; dtype=float64 gives the weights of
    exact arithmetic.  At non-dyadic scales the two differ by up to ~2.5e-6 (37 -> 96).  (The rows lie along the
    width: aten's CPU antialias kernel resizes a [.., n, 1] image along its height wrongly.)"""
    eye = torch.eye(n_in, dtype=dtype).reshape(1, n_in, 1, n_in)
    up = F.interpolate(eye, size=(1, n_out), mode="bilinear", align_corners=False, antialias=True)
    return up.reshape(n_in, n_out).t().to(device=device, dtype=torch.float64).contiguous()


def project64(masks: torch.Tensor, enc_hw, chunk: int = 128, weights=torch.float32) -> torch.Tensor:
    """proj64 [n, eh*ew] float64 = Uy^T M Ux of the thresholded masks (`ref_torch.threshold_lowres`): the reference's
    masks @ upsample(feat) is (masks @ U) @ feat with the separable U = Uy (x) Ux.  The weights are the reference's
    (`axis_weights`, float32 recipe by default); everything after them is float64.  Computed on masks.device in chunks
    (the dense [P, E] operator does not fit in float64)."""
    n, h, w = masks.shape
    eh, ew = enc_hw
    uy, ux = axis_weights(eh, h, masks.device, weights), axis_weights(ew, w, masks.device, weights)
    out = torch.empty((n, eh * ew), dtype=torch.float64, device=masks.device)
    for i in range(0, n, chunk):
        m = ref_torch.threshold_lowres(masks[i:i + chunk]).to(torch.float64).reshape(-1, h, w)
        out[i:i + chunk] = (uy.t() @ (m @ ux)).reshape(m.shape[0], eh * ew)
    return out


def pooled64(proj64: torch.Tensor, feat64: torch.Tensor, area: torch.Tensor):
    """-> (obj64, bound): F.normalize((proj feat) / area) and the per-element error scale of a normalised pooled row,
    (|proj| |feat|) / area / ||(proj feat) / area|| (0 on rows whose reference is zero)."""
    a = area.to(torch.float64).clamp(min=1.0).unsqueeze(1)
    s = (proj64 @ feat64) / a
    nrm = s.norm(dim=1, keepdim=True)
    obj = s / nrm.clamp(min=1e-12)
    bound = ((proj64.abs() @ feat64.abs()) / a) / torch.where(nrm > 0, nrm, torch.ones_like(nrm))
    return obj, bound


def normalised_error(got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, what: str) -> float:
    """max |got - ref| / bound over the elements with bound > 0; elements with bound == 0 (their reference is an exact
    zero: empty masks, zero rows) must be exact zeros."""
    got, ref, bound = got.to(torch.float64), ref.to(torch.float64), bound.to(ref.device, torch.float64)
    got = got.to(ref.device)
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    zero = bound == 0
    if zero.any():
        assert (ref[zero] == 0).all()
        assert (got[zero] == 0).all(), f"{what}: {int((got[zero] != 0).sum())} elements of zero rows are not zero"
    live = ~zero
    if not live.any():
        return 0.0
    return float(((got - ref).abs()[live] / bound[live]).max())


def check_labels(sim_got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, what: str, labels=None):
    """Top-1 labels: exactly the argmax of the kernel's own sim (lowest index on ties), and the float64 argmax except
    where the float64 top-2 gap lies inside the row's band of 2 * TOL_SIM * max bound."""
    sim_got = sim_got.to(torch.float64)
    own = sim_got.argmax(1)
    if labels is not None:
        assert torch.equal(labels.to(own.device, torch.int64), own), f"{what}: top_label is not the argmax of sim"
    want = ref.argmax(1)
    bad = torch.nonzero(own.to(want.device) != want).flatten()
    if bad.numel():
        own = own.to(want.device)
        gap = ref[bad, want[bad]] - ref[bad, own[bad]]
        band = 2 * TOL_SIM * bound[bad].max(dim=1).values
        assert (gap <= band).all(), f"{what}: label differs from the float64 argmax outside the tolerance band"
    return int(bad.numel())
