"""CPU ORACLE OF THE DDIM SAMPLER -- TEST INFRASTRUCTURE ONLY.

The reference has no DDIM sampler, so this restates improved_diffusion/gaussian_diffusion.py: ddim_sample / ddim_sample_loop
(DiT diffusion/gaussian_diffusion.py: ddim_sample) with clip_denoised=False, on top of the reference restatement in
oracle/restate.py (linear betas, respacing, denoiser forward).  Parity is UNPINNED against the reference; tests/test_ddim.py
ties it to the reference-pinned DDPM tables through the eta = 1 identity (sigma^2 = posterior variance, mean = posterior mean).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import restate as R


def kept_timesteps(spacing, diffusion_steps: int = 1000):
    """respace.py:12-62 for one section given as an int count, or a "ddimN" string (the smallest integer stride giving
    exactly N steps)."""
    if isinstance(spacing, str) and spacing.startswith("ddim"):
        want = int(spacing[4:])
        for stride in range(1, diffusion_steps):
            if len(range(0, diffusion_steps, stride)) == want:
                return list(range(0, diffusion_steps, stride))
        raise ValueError(f"cannot create exactly {want} steps with an integer stride")
    return R.kept_timesteps(int(spacing), diffusion_steps)


def schedule(spacing, diffusion_steps: int = 1000):
    """float64 tables of the respaced linear schedule (as R.respaced_schedule builds them) that ddim_sample reads."""
    scale = 1000 / diffusion_steps
    base_ac = np.cumprod(1.0 - np.linspace(scale * 0.0001, scale * 0.02, diffusion_steps, dtype=np.float64))
    keep = set(kept_timesteps(spacing, diffusion_steps))
    last, betas, tmap = 1.0, [], []
    for i, ac in enumerate(base_ac):
        if i in keep:
            betas.append(1 - ac / last)
            last = ac
            tmap.append(i)
    betas = np.array(betas, dtype=np.float64)
    ac = np.cumprod(1.0 - betas, axis=0)
    return {"timestep_map": np.array(tmap, dtype=np.int64), "betas": betas, "sqrt_recip_ac": np.sqrt(1.0 / ac),
            "sqrt_recipm1_ac": np.sqrt(1.0 / ac - 1), "alphas_cumprod": ac, "alphas_cumprod_prev": np.append(1.0, ac[:-1])}


def ddim_terms(x, eps, step, sched, eta):
    """ddim_sample up to the noise term: (pred_xstart, mean_pred, sigma).  The tables are taken as IDDPM's
    _extract_into_tensor takes them (float64 -> x.dtype, i.e. fp32 for fp32 inputs) and every later operation runs in that
    dtype in IDDPM's order."""
    tab = lambda name: torch.tensor(float(sched[name][step]), dtype=x.dtype)        # one rounding of the float64 entry
    pred_xstart = tab("sqrt_recip_ac") * x - tab("sqrt_recipm1_ac") * eps                # _predict_xstart_from_eps
    eps = (tab("sqrt_recip_ac") * x - pred_xstart) / tab("sqrt_recipm1_ac")             # _predict_eps_from_xstart
    alpha_bar, alpha_bar_prev = tab("alphas_cumprod"), tab("alphas_cumprod_prev")
    sigma = eta * torch.sqrt((1 - alpha_bar_prev) / (1 - alpha_bar)) * torch.sqrt(1 - alpha_bar / alpha_bar_prev)
    mean_pred = pred_xstart * torch.sqrt(alpha_bar_prev) + torch.sqrt(1 - alpha_bar_prev - sigma ** 2) * eps
    return pred_xstart, mean_pred, sigma


def ddim_update(x, model_out, step, noise, sched, eta):
    """One DDIM step: mean_pred + [step != 0] sigma noise; `noise` may be None when eta = 0."""
    C = x.shape[-1]
    _, mean_pred, sigma = ddim_terms(x, model_out[..., :C], step, sched, eta)
    if noise is None:
        assert eta == 0, "eta > 0 needs noise"
        return mean_pred
    return mean_pred + (0.0 if step == 0 else 1.0) * sigma * noise


def sample_loop(sd, z, X, cg_z, mask, noises, sched, eta, k_neighbors=64):
    """ddim_sample_loop through _WrappedModel's timestep remap (respace.py:117-129), the denoiser being the oracle's
    (R.denoiser_forward, features hoisted as R.sample_loop does).  noises[s] is the N(0,1) draw of respaced step s; None at eta = 0."""
    g = R.edge_embedding(sd, X, mask.to(torch.int32), k_neighbors)
    graph = (g[0], g[3])
    x = z
    for s in list(range(len(sched["betas"])))[::-1]:
        t = torch.full((x.shape[0],), int(sched["timestep_map"][s]), dtype=torch.int64)
        out = R.denoiser_forward(sd, x, t, X, cg_z, mask, k_neighbors, graph=graph)
        x = ddim_update(x, out, s, None if noises is None else noises[s], sched, eta)
    return x
