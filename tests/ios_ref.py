"""Exact and float64 references of the intersection-over-self term (compute_semantic_ios,
matching_baseline_utils.py:831-867), shared by the IoS accuracy tests.  The module docstring of
test_ios_decay_accuracy.py defines the metric and says how the tolerances were set."""
import torch

TOL_IOS = 4e-7        # normalised IoS error limit of the kernels (module docstring)
TOL_REF_IOS = 1.2e-6  # the same for the reference's own fp32 values stored in the golden files
RESOLUTION_PX = 1.0   # TOL_IOS * bound_i, in pixels of s^2 / area_i, must stay below this in every intersecting row
INTER_SLICE = 1 << 18  # pixels per fp32 product slice (partial sums < 2^24: exact)


def inter_counts(masks: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """masks [K, ...] bool, labels [K] -> int64 [K, K]: exact same-label intersection counts, 0 on the diagonal and
    across labels.  Per label group, fp32 products with TF32 off in slices of INTER_SLICE pixels (exact integers)."""
    k = masks.shape[0]
    flat = masks.reshape(k, -1)
    labels = labels.to(flat.device)
    out = torch.zeros((k, k), dtype=torch.int64, device=flat.device)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for lab in torch.unique(labels).tolist():
            idx = torch.nonzero(labels == lab).flatten()
            if idx.numel() < 2:
                continue
            acc = torch.zeros((idx.numel(), idx.numel()), dtype=torch.int64, device=flat.device)
            for p0 in range(0, flat.shape[1], INTER_SLICE):
                m = flat[idx, p0:p0 + INTER_SLICE].to(torch.float32)
                acc += (m @ m.t()).round().to(torch.int64)
            out[idx.unsqueeze(1), idx.unsqueeze(0)] = acc
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    out.fill_diagonal_(0)
    return out


def ios_reference(inter: torch.Tensor, area: torch.Tensor, feats: torch.Tensor, labels: torch.Tensor):
    """-> (ios64 [K], bound [K], s2_per_px [K]) in float64: the reference's row maximum
    max_{j != i, same label} ((inter * s) / area_i) * s with s = max(f_i . f_j, 0), 0 for rows without an intersecting
    partner and for area-0 rows (the tap's value before the empty-mask rule); the row's error bound
    max_j (inter / area_i) (2 s sum|f_i f_j| + s^2); and s^2 / area_i of the maximising partner (what one pixel of
    intersection moves the row by)."""
    dev = inter.device
    f = feats.to(device=dev, dtype=torch.float64)
    s = (f @ f.t()).clamp(min=0.0)
    a = f.abs() @ f.abs().t()
    labels = labels.to(dev)
    same = labels.unsqueeze(1) == labels.unsqueeze(0)
    same.fill_diagonal_(False)
    ar = area.to(device=dev, dtype=torch.float64).clamp(min=1.0).unsqueeze(1)
    it = inter.to(torch.float64) * same
    v = ((it * s) / ar) * s
    b = (it / ar) * (2.0 * s * a + s * s)
    if v.shape[0] == 0:
        z = torch.zeros(0, dtype=torch.float64, device=dev)
        return z, z, z
    ios, j = v.max(dim=1)
    bound = b.max(dim=1).values
    s_best = s.gather(1, j.unsqueeze(1)).squeeze(1)
    empty = area.to(dev) == 0
    ios[empty], bound[empty] = 0.0, 0.0
    return ios, bound, s_best * s_best / ar.squeeze(1)


def ios_errors(got: torch.Tensor, ios64, bound, s2_per_px, what: str):
    """-> (largest normalised error, largest tolerance in pixels).  Rows whose bound is 0 must be exact zeros."""
    got = got.to(ios64.device, torch.float64)
    assert torch.isfinite(got).all(), f"{what}: non-finite IoS in the tap"
    zero = bound == 0
    assert (ios64[zero] == 0).all()
    assert (got[zero] == 0).all(), f"{what}: {int((got[zero] != 0).sum())} rows without a partner are not 0"
    live = ~zero
    if not live.any():
        return 0.0, 0.0
    err = float(((got - ios64).abs()[live] / bound[live]).max())
    hit = live & (ios64 > 0)
    px = float((TOL_IOS * bound[hit] / s2_per_px[hit]).max()) if hit.any() else 0.0
    return err, px
