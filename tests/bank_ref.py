"""Float64 and exact references of the memory-bank fill, its post-processing, the prototypes and the negative-reference
scoring (csrc/fill.cu, csrc/score.cu), shared by the bank accuracy tests.  The module docstring of
test_bank_accuracy.py defines the metrics and says how the tolerances were set."""
import math

import numpy as np
import torch

from gemm_ref import TOL_SIM

U = 2.0 ** -24  # unit roundoff of fp32


def gamma(n: int) -> float:
    """Higham's gamma_n = n u / (1 - n u): the relative error bound of n fp32 roundings in a chain."""
    return n * U / (1.0 - n * U)


def tol_fill(e: int) -> float:
    """fill_pool_kernel: per output column ceil(E/8) fmas in one warp, then the 8 warp partials added in order."""
    return gamma(math.ceil(e / 8) + 8)


def tol_wsum(e: int) -> float:
    """fill_pool_kernel: the weight sum is ceil(E/32) adds per lane, then a 5-level butterfly."""
    return gamma(math.ceil(e / 32) + 5)


def tol_proto(shots: int, c: int) -> float:
    """proto_prepare_kernel: `shots` adds and one division for the mean, ceil(c/32) fmas and a 5-level butterfly for the
    squared norm, one square root, one division."""
    return gamma(shots + 1 + math.ceil(c / 32) + 5 + 1 + 1)


def nearest_index(dst, in_size: int, out_size: int) -> np.ndarray:
    """aten's nearest source index (upsample_nearest: `min(floorf(dst * ((float)in / out)), in - 1)`) with its fp32
    rounding, and its shortcuts for out == in and out == 2 in (which agree with the formula).  dst: int or array."""
    dst = np.asarray(dst, dtype=np.int64)
    if in_size == out_size:
        return dst.copy()
    if out_size == 2 * in_size:
        return dst >> 1
    scale = np.float32(in_size) / np.float32(out_size)
    src = np.floor(dst.astype(np.float32) * scale).astype(np.int64)
    return np.minimum(src, in_size - 1)


def exact_nearest_index(dst, in_size: int, out_size: int) -> np.ndarray:
    """floor(dst * in / out) in integer arithmetic: what the fp32 formula approximates."""
    dst = np.asarray(dst, dtype=np.int64)
    return np.minimum(dst * in_size // out_size, in_size - 1)


def gather_lowres(soft: torch.Tensor, enc_hw) -> torch.Tensor:
    """soft [b, mh, mw] -> [b, eh*ew]: the nearest-resized soft masks (F.interpolate(mode="nearest"))."""
    b, mh, mw = soft.shape
    eh, ew = enc_hw
    iy = torch.from_numpy(nearest_index(np.arange(eh), mh, eh)).to(soft.device)
    ix = torch.from_numpy(nearest_index(np.arange(ew), mw, ew)).to(soft.device)
    return soft[:, iy][:, :, ix].reshape(b, eh * ew)


def fill64(feat: torch.Tensor, soft: torch.Tensor, enc_hw):
    """feat [b, E, C] fp32, soft [b, mh, mw] fp32 -> (sum64 [b, C], wsum64 [b], mask_lowres [b, E] fp32, bound [b, C],
    wbound [b]): sum_e m_e f_e and sum_e m_e in float64, the gathered soft mask, sum_e |m_e| |f_e| and sum_e |m_e|."""
    m = gather_lowres(soft, enc_hw)
    m64, f64 = m.to(torch.float64), feat.to(torch.float64)
    sum64 = torch.bmm(m64.unsqueeze(1), f64).squeeze(1)
    bound = torch.bmm(m64.abs().unsqueeze(1), f64.abs()).squeeze(1)
    return sum64, m64.sum(1), m, bound, m64.abs().sum(1)


def finalize32(feats_sum: torch.Tensor, mask_sum: torch.Tensor):
    """fill_finalize_kernel restated in fp32 with IEEE operations in the kernel's order: feats_sum [n_cls, L, C],
    mask_sum [n_cls, L] -> (ins_avg [n_cls, L, C], avg [n_cls, C]).  The per-slot and the class weights are summed over
    l in order from 0.0f, a zero weight is replaced by 1, each division is correctly rounded."""
    s, w = feats_sum.to(torch.float32), mask_sum.to(torch.float32)
    n_cls, shots, c = s.shape
    wall = torch.zeros((n_cls,), dtype=torch.float32, device=s.device)
    tot = torch.zeros((n_cls, c), dtype=torch.float32, device=s.device)
    for l in range(shots):
        wall = wall + w[:, l]
        tot = tot + s[:, l]
    one = torch.ones_like(w)
    ins_avg = s / torch.where(w == 0, one, w).unsqueeze(-1)
    avg = tot / torch.where(wall == 0, torch.ones_like(wall), wall).unsqueeze(-1)
    return ins_avg, avg


def proto64(ins_avg: torch.Tensor):
    """ins_avg [n_cls, L, C] -> (proto64 [n_cls, C], bound [n_cls, C]): the mean over all L slots (unfilled zeros
    included), L2-normalised, in float64.  The first-order error of the kernel's fp32 arithmetic is at most
    tol_proto(L, C) * bound with bound_i = (S_i + |p_i| ||S||) / ||m|| + |p_i|, S = mean_l |x_l| (the sum's error scale,
    also moving the norm) and |p_i| for the relative errors of the norm and the divisions.  0 on zero rows."""
    x = ins_avg.to(torch.float64)
    m = x.mean(dim=1)
    s = x.abs().mean(dim=1)
    nrm = m.norm(dim=1, keepdim=True)
    live = nrm > 0
    p = m / torch.where(live, nrm, torch.ones_like(nrm))
    bound = (s + p.abs() * s.norm(dim=1, keepdim=True)) / torch.where(live, nrm, torch.ones_like(nrm)) + p.abs()
    return p, torch.where(live, bound, torch.zeros_like(bound))


def neg_terms(obj: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, l_neg: int):
    """float64 (sp_raw [n, n_cls], sn_all [n, n_cls, l_neg] clamped at 0, a_pos [n, n_cls], a_neg [n, n_cls, l_neg]):
    the two similarity products and their GEMM error scales |obj| |proto|^T."""
    o, p, q = obj.to(torch.float64), pos.to(torch.float64), neg.to(torch.float64)
    n, n_cls = o.shape[0], p.shape[0]
    sp = o @ p.t()
    sn = (o @ q.t()).clamp(min=0.0).reshape(n, n_cls, l_neg)
    a_pos = o.abs() @ p.abs().t()
    a_neg = (o.abs() @ q.abs().t()).reshape(n, n_cls, l_neg)
    return sp, sn, a_pos, a_neg


def neg_formula(sp_raw, sn, sigma: float, clamp_pos=True, div_sigma=True):
    """sim = sp * exp(-clamp(sn - sp, 0) / sigma) with sp = clamp(sp_raw, 0) (ref_torch.pool_and_score_neg).  The two
    switches emulate defects: no clamp on sim_pos, multiplying by sigma instead of dividing."""
    sp = sp_raw.clamp(min=0.0) if clamp_pos else sp_raw
    d = (sn - sp).clamp(min=0.0)
    return sp * torch.exp(-d / sigma if div_sigma else -d * sigma)


def neg64(obj: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, l_neg: int, sigma: float):
    """-> (sim64 [n, n_cls], bound [n, n_cls]): negative-reference scoring in float64 and the scale B of the kernel's
    error, |got - sim64| <= TOL_SIM * B.  B propagates the GEMM errors (TOL_SIM |obj| |proto|^T per product) to first
    order, (1 + sp/sigma) |obj||pos|^T + (sp/sigma) max_l |obj||neg_l|^T, and adds the fp32 roundings after the GEMMs:
    (2x + 8) u |sim64| / TOL_SIM for x = clamp(sn - sp, 0) / sigma (the subtraction and the division, amplified by exp,
    expf's 2 ulps and the final product)."""
    sp_raw, sn_all, a_pos, a_neg = neg_terms(obj, pos, neg, l_neg)
    sn = sn_all.max(dim=-1).values
    sim = neg_formula(sp_raw, sn, sigma)
    sp = sp_raw.clamp(min=0.0)
    x = (sn - sp).clamp(min=0.0) / sigma
    bound = (1.0 + sp / sigma) * a_pos + (sp / sigma) * a_neg.max(dim=-1).values \
        + (2.0 * x + 8.0) * U * sim.abs() / TOL_SIM
    return sim, bound
