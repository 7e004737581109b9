"""CPU ORACLE OF LATENT INPAINTING -- TEST INFRASTRUCTURE ONLY.

Restates the replacement method for inpainting with a diffusion model on top of the DDPM restatement in oracle/restate.py
(p_sample_update, denoiser_forward) and the DDIM restatement in tests/ddim_oracle.py.  With eps = z on the kept rows:
  1. before the first step every kept row is set to sqrt(acp[T-1]) x0 + sqrt(1 - acp[T-1]) eps;
  2. at every respaced step s = T-1 .. 0 every row gets the unchanged update, then every kept row is overwritten with
     sqrt(acp_prev[s]) x0 + sqrt(1 - acp_prev[s]) eps (acp_prev[0] = 1, so kept rows end at x0).
The levels are fp32 roundings of float64 values, and a * x0 + b * eps is two rounded fp32 products and one rounded sum.
Parity is UNPINNED against any reference (the reference has no inpainting); tests/test_inpaint.py ties it to the pinned
oracle through the all-False identity (no kept row: exactly R.sample_loop / D.sample_loop).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import restate as R
from tests import ddim_oracle as D


def level_table(spacing, diffusion_steps: int = 1000):
    """[T+1, 2] fp32: rows s < T {sqrt(acp_prev[s]), sqrt(1 - acp_prev[s])}, row T {sqrt(acp[T-1]), sqrt(1 - acp[T-1])}."""
    s = D.schedule(spacing, diffusion_steps)
    level = np.append(s["alphas_cumprod_prev"], s["alphas_cumprod"][-1])
    return torch.from_numpy(np.stack([np.sqrt(level), np.sqrt(1.0 - level)], axis=1).astype(np.float32))


def sample_loop(sd, z, X, cg_z, mask, noises, spacing, keep, x0, sampler="ddpm", eta=0.0, k_neighbors=64):
    """The DDPM (R.sample_loop) or DDIM (D.sample_loop, `eta`) loop of respacing `spacing` with the rows where keep [B,L] is
    True following x0 [B,L,3].  noises[s] is the N(0,1) draw of respaced step s (None for DDIM at eta = 0)."""
    q = level_table(spacing)
    T = q.shape[0] - 1
    sched = R.respaced_schedule(int(spacing)) if sampler == "ddpm" else D.schedule(spacing)
    g = R.edge_embedding(sd, X, mask.to(torch.int32), k_neighbors)
    graph = (g[0], g[3])
    kept = keep[..., None]
    eps = z
    level = lambda r: q[r, 0] * x0 + q[r, 1] * eps
    x = torch.where(kept, level(T), z)
    for s in list(range(T))[::-1]:
        t = torch.full((x.shape[0],), int(sched["timestep_map"][s]), dtype=torch.int64)
        out = R.denoiser_forward(sd, x, t, X, cg_z, mask, k_neighbors, graph=graph)
        if sampler == "ddpm":
            x = R.p_sample_update(x, out, s, noises[s], sched)
        else:
            x = D.ddim_update(x, out, s, None if noises is None else noises[s], sched, eta)
        x = torch.where(kept, level(s), x)
    return x
