"""CPU ORACLE OF PARTIAL-NOISE REFINEMENT -- TEST INFRASTRUCTURE ONLY.

Restates partial-noise refinement (SDEdit) with latent inpainting on top of the DDPM restatement in oracle/restate.py, the DDIM
restatement in tests/ddim_oracle.py and the inpainting level table of tests/inpaint_oracle.py.  For a start of `steps` respaced
steps, with eps = z on every row:
  1. before the first step EVERY row, kept or not, is set to level[steps] = sqrt(acp[steps-1]) x0 + sqrt(1 - acp[steps-1]) eps;
  2. at every respaced step s = steps-1 .. 0 every row gets the unchanged update, then every kept row is overwritten with
     level[s] (level[0] = x0, so kept rows end at x0).
a * x0 + b * eps is two rounded fp32 products and one rounded sum, as in the inpainting oracle.  Parity is UNPINNED against any
reference (the reference has no refinement); tests/test_refine.py ties it to the pinned oracle: with steps = T and no kept row it
is R.sample_loop / D.sample_loop started from level[T].
"""
from __future__ import annotations

import torch

from oracle import restate as R
from tests import ddim_oracle as D
from tests import inpaint_oracle as I


def sample_loop(sd, z, X, cg_z, mask, noises, spacing, steps, keep, x0, sampler="ddpm", eta=0.0, k_neighbors=64):
    """Refine x0 [B,L,3] over the last `steps` respaced steps of the DDPM (R) or DDIM (D, `eta`) loop of respacing `spacing`, the
    rows where keep [B,L] is True following x0.  noises[s] is the N(0,1) draw of respaced step s (None for DDIM at eta = 0)."""
    q = I.level_table(spacing)
    T = q.shape[0] - 1
    assert 1 <= steps <= T
    sched = R.respaced_schedule(int(spacing)) if sampler == "ddpm" else D.schedule(spacing)
    g = R.edge_embedding(sd, X, mask.to(torch.int32), k_neighbors)
    graph = (g[0], g[3])
    kept = keep[..., None]
    level = lambda r: q[r, 0] * x0 + q[r, 1] * z
    x = level(steps)
    for s in list(range(steps))[::-1]:
        t = torch.full((x.shape[0],), int(sched["timestep_map"][s]), dtype=torch.int64)
        out = R.denoiser_forward(sd, x, t, X, cg_z, mask, k_neighbors, graph=graph)
        if sampler == "ddpm":
            x = R.p_sample_update(x, out, s, noises[s], sched)
        else:
            x = D.ddim_update(x, out, s, None if noises is None else noises[s], sched, eta)
        x = torch.where(kept, level(s), x)
    return x
