"""Step-3 chain statistics on the device, for batches too large to leave it as text.

Restates, with torch ops on the chain tensor the sampler produced ([rows, walkers, P+1], float64):
separation and position angle (apf_step3.py:255-256,283-291, without the distortion lookup whose
FITS tables are absent from the checkout), their median / 68% interval (:436-437 uses median and
std), and Gelman-Rubin per parameter (:260-278) -- per frame, since one batch holds many epochs.
"""
from __future__ import annotations

import math

import torch

from .chains import PIXSCALE_PRE2015

Q68 = (0.15865, 0.5, 0.84135)


def separation_pa(chain, pixscale=PIXSCALE_PRE2015, companion=1):
    """sep [mas] and pa [deg] of object ``companion`` relative to the star, for every row and walker."""
    dx = chain[..., 2 * companion] - chain[..., 0]
    dy = chain[..., 2 * companion + 1] - chain[..., 1]
    sep = torch.sqrt(dx * dx + dy * dy) * pixscale
    pa = torch.rad2deg(torch.atan2(-dx, dy))
    return sep, pa


def per_frame_summary(chain, frame_of, n_frames, pixscale=PIXSCALE_PRE2015, companion=1):
    """For each frame: quantiles (16, 50, 84 %) and std of sep and pa pooled over that frame's
    walkers and all rows.  Returns a dict of [n_frames, 3] / [n_frames] float64 tensors."""
    sep, pa = separation_pa(chain, pixscale, companion)
    frame_of = torch.as_tensor(frame_of, device=chain.device).long()
    q = torch.tensor(Q68, dtype=torch.float64, device=chain.device)
    out = {k: [] for k in ("sep_q", "pa_q", "sep_std", "pa_std", "walkers")}
    for f in range(n_frames):
        sel = frame_of == f
        s, p = sep[:, sel].reshape(-1), pa[:, sel].reshape(-1)
        out["walkers"].append(int(sel.sum()))
        if s.numel() == 0:
            nan = torch.full((3,), float("nan"), dtype=torch.float64, device=chain.device)
            out["sep_q"].append(nan); out["pa_q"].append(nan)
            out["sep_std"].append(nan[0]); out["pa_std"].append(nan[0])
            continue
        out["sep_q"].append(torch.quantile(s, q)); out["pa_q"].append(torch.quantile(p, q))
        out["sep_std"].append(s.std(unbiased=False)); out["pa_std"].append(p.std(unbiased=False))
    return {"sep_q": torch.stack(out["sep_q"]), "pa_q": torch.stack(out["pa_q"]),
            "sep_std": torch.stack(out["sep_std"]), "pa_std": torch.stack(out["pa_std"]),
            "walkers": torch.tensor(out["walkers"])}


def gelman_rubin(chain_cols, python2_division=True):
    """apf_step3.py:262-276 for [rows, walkers, columns] at once -> (PSRF, RC), each [columns]."""
    n, m = float(chain_cols.shape[0]), float(chain_cols.shape[1])
    w = chain_cols.var(dim=0, unbiased=False).sum(dim=0) / m
    means = chain_cols.mean(dim=0)
    b = (n / (m - 1.0)) * ((means - means.mean(dim=0, keepdim=True)) ** 2).sum(dim=0)
    psrf = (((n - 1.0) / n) * w + ((m + 1.0) / (m * n)) * b) / w
    factor = 1.0 if python2_division else 19.0 / 17.0
    return psrf, torch.sqrt(factor * psrf)


# ----------------------------------------------------------------------------------------------
# Monte Carlo error from the on-device batch means (lapf_sampler_batchmeans): no chain needed
# ----------------------------------------------------------------------------------------------
def batch_means_summary(bm, walkers_per_frame, rows, min_batches=20):
    """Per frame and quantity, from ``GibbsSampler.batch_means()`` (its ``frame`` sums and the walker
    counts all-reduced over ranks if the walkers are sharded) with M walkers of ``rows`` rows each:
    the largest batch length b = batch_rows * 2^l with J = rows // b >= ``min_batches`` complete
    batches is used; with s2 the mean over walkers of the sample variance of their batch means and
    sigma2 the mean of their row variances,
        tau = b * s2 / sigma2  (integrated autocorrelation time, rows),  ess = M * rows / tau,
        mcse = sqrt(s2 / (J * M))  (standard error of the mean pooled over the frame's walkers).
    Returns a dict of float64 tensors: tau, ess, mcse [F, C] (nan where no level qualifies),
    tau_levels [F, C, levels] (nan at the levels with fewer than ``min_batches`` batches: a reader
    sees whether tau has levelled off), batch_rows_used (int, or None if no level qualifies)."""
    frame = torch.as_tensor(bm["frame"], dtype=torch.float64)
    b0, levels, rows = int(bm["batch_rows"]), int(bm["levels"]), int(rows)
    m = torch.as_tensor(walkers_per_frame, dtype=torch.float64, device=frame.device).reshape(-1, 1)
    sigma2 = frame[..., 0] / m
    nan = torch.full_like(sigma2, float("nan"))
    tau_levels, use = [], None
    for lv in range(levels):
        b = b0 << lv
        if rows // b >= min_batches:
            tau_levels.append(b * (frame[..., 1 + lv] / m) / sigma2)
            use = lv
        else:
            tau_levels.append(nan)
    if use is None:
        return {"tau": nan, "ess": nan.clone(), "mcse": nan.clone(), "tau_levels": torch.stack(tau_levels, dim=-1),
                "batch_rows_used": None}
    b = b0 << use
    j = rows // b
    s2 = frame[..., 1 + use] / m
    tau = b * s2 / sigma2
    return {"tau": tau, "ess": m * rows / tau, "mcse": torch.sqrt(s2 / (j * m)),
            "tau_levels": torch.stack(tau_levels, dim=-1), "batch_rows_used": b}


# ----------------------------------------------------------------------------------------------
# the same summary from the on-device sketches (lapf_sampler_sketch): no chain needed
# ----------------------------------------------------------------------------------------------
def quantiles_from_hist(hist, center, bin_width, q=Q68):
    """Quantiles of a fixed-bin histogram [..., n_bins + 2] (bin 0: below range, last: above) whose bin
    n_bins/2 starts at ``center`` [...]; linear inside the bin, so exact to the bin width.  Returns
    [..., len(q)] float64; nan where a quantile falls into an out-of-range bin or nothing was recorded."""
    hist = torch.as_tensor(hist).double()
    center = torch.as_tensor(center, dtype=torch.float64, device=hist.device)
    n_bins = hist.shape[-1] - 2
    cum = hist.cumsum(dim=-1)
    total = cum[..., -1:]
    out = []
    for qq in q:
        target = qq * total                                             # [..., 1]
        idx = (cum < target).sum(dim=-1, keepdim=True).clamp(max=n_bins + 1)   # first bin with cum >= target
        below = torch.where(idx > 0, cum.gather(-1, (idx - 1).clamp(min=0)), torch.zeros_like(target))
        inside = hist.gather(-1, idx).clamp(min=1.0)
        frac = ((target - below) / inside).clamp(0.0, 1.0)
        val = center.unsqueeze(-1) + ((idx - 1 - n_bins // 2).double() + frac) * bin_width
        bad = (idx < 1) | (idx > n_bins) | (total <= 0)
        out.append(torch.where(bad, torch.full_like(val, float("nan")), val))
    return torch.cat(out, dim=-1)


def sketch_summary(sk, pixscale=PIXSCALE_PRE2015):
    """Per frame and companion, from ``GibbsSampler.sketch()`` (all-reduced over ranks if the walkers
    are sharded): separation [mas] and position angle [deg] quantiles (16, 50, 84 %), mean and
    standard deviation -- what apf_step3.py:436-437 reports (median, std) -- plus the fraction of
    recorded values outside the histogram range.  Returns a dict of [F, nbody-1, ...] tensors."""
    hist, summ = sk["hist"], sk["summary"]
    center, s1, s2, n = summ[..., 0], summ[..., 1], summ[..., 2], summ[..., 3].clamp(min=1.0)
    width = torch.tensor([sk["sep_bin"], sk["pa_bin"]], dtype=torch.float64, device=hist.device)
    qs = quantiles_from_hist(hist, center, width.view(1, 1, 2, 1).expand(hist.shape[:-1] + (1,)))
    mean = center + s1 / n
    std = torch.sqrt((s2 / n - (s1 / n) ** 2).clamp(min=0.0))
    scale = torch.tensor([pixscale, 1.0], dtype=torch.float64, device=hist.device)
    tot = hist.sum(dim=-1).clamp(min=1)
    outside = (hist[..., 0] + hist[..., -1]).double() / tot.double()
    return {"sep_q": qs[..., 0, :] * pixscale, "pa_q": qs[..., 1, :],
            "sep_mean": mean[..., 0] * pixscale, "pa_mean": mean[..., 1],
            "sep_std": std[..., 0] * pixscale, "pa_std": std[..., 1],
            "outside": outside, "count": summ[..., 0, 3], "scale": scale}
