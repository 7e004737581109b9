"""Deterministic synthetic inputs for the sampling path (SURVEY.md section 8d).

Produces the same batch-dict schema the reference's data pipeline hands to the hot path
(`build_ic_peptide_dataset`, utils/protein_module.py:782-869 + `CG_collate`,
utils/dataset_module.py:259-295), restricted to the keys the path reads:
CG_nxyz, OG_CG_nxyz, num_CGs, num_atoms, CG_nbr_list, prot_idx; plus `info_dict`.
All generators are seeded CPU torch generators so the CPU oracle and the CUDA path see
bit-identical inputs.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import topology

CG_CUTOFF = 21.0  # utils/model_module.py:23


def ca_trace(num_frames: int, num_res_with_termini: int, seed: int, compact: float = 0.0) -> torch.Tensor:
    """Freely-jointed C-alpha walk with jittered bond length U(3.70, 3.90) Angstrom (keeps the
    3.6 < |dX| < 4.0 gate of protein_mpnn_utils.py:400 open and avoids exact distance ties).
    `compact` > 0 adds a weak pull towards the running centroid ("Atlas-like" globule)."""
    g = torch.Generator().manual_seed(seed)
    n = num_res_with_termini
    d = torch.randn(num_frames, n, 3, generator=g)
    b = 3.70 + 0.20 * torch.rand(num_frames, n, 1, generator=g)
    if compact <= 0.0:
        d = b * d / d.norm(dim=-1, keepdim=True)
        return torch.cumsum(d, dim=1)
    X = torch.zeros(num_frames, n, 3)
    pos = torch.zeros(num_frames, 3)
    cen = torch.zeros(num_frames, 3)
    for i in range(n):
        step = d[:, i] + compact * (cen - pos)
        step = b[:, i] * step / step.norm(dim=-1, keepdim=True)
        pos = pos + step
        X[:, i] = pos
        cen = cen + (pos - cen) / (i + 1)
    return X


def radius_graph(xyz: torch.Tensor, cutoff: float = CG_CUTOFF) -> torch.Tensor:
    """Undirected (i < j) neighbour list within `cutoff` (utils/protein_module.py:567-584)."""
    n = xyz.shape[0]
    diff = xyz[None, :, :] - xyz[:, None, :]
    dist = diff.pow(2).sum(dim=2).sqrt()
    keep = dist <= cutoff
    keep[torch.arange(n), torch.arange(n)] = False
    nbr = torch.nonzero(keep)
    return nbr[nbr[:, 1] > nbr[:, 0]]


@dataclass
class SyntheticProtein:
    """One protein (one topology) with `num_frames` conformations."""
    restype_full: torch.Tensor   # [L+2] int64, termini included
    ca_full: torch.Tensor        # [F, L+2, 3] fp32
    info: tuple                  # (permute, atom_idx, atom_orders)

    @property
    def L(self) -> int:
        return self.restype_full.numel() - 2

    @property
    def num_atoms(self) -> int:
        return int(self.info[0].numel())


def make_protein(L: int, num_frames: int, seed: int, compact: float = 0.0) -> SyntheticProtein:
    g = torch.Generator().manual_seed(seed + 7919)
    restype = torch.randint(0, 20, (L + 2,), generator=g)
    X = ca_trace(num_frames, L + 2, seed, compact)
    return SyntheticProtein(restype, X, topology.build_info(restype[1:-1]))


def trajectory(L: int, num_frames: int, seed: int, step: float = 0.05, compact: float = 0.0) -> SyntheticProtein:
    """One protein whose C-alpha trace moves from frame to frame by a Gaussian step of RMS length `step` Angstrom per residue
    (a random walk from make_protein's first frame), like consecutive frames of an MD trajectory."""
    prot = make_protein(L, 1, seed, compact)
    g = torch.Generator().manual_seed(seed + 104729)
    moves = torch.randn(num_frames - 1, L + 2, 3, generator=g) * (step / 3 ** 0.5)
    ca = prot.ca_full[0] + torch.cat([torch.zeros(1, L + 2, 3), torch.cumsum(moves, 0)])
    return SyntheticProtein(prot.restype_full, ca, prot.info)


def collate(protein: SyntheticProtein, frames=None, prot_idx: int = 0) -> dict:
    """Batch dict for `frames` of one protein, exactly the keys/shapes the reference hot path
    indexes (models/latent_model.py:168-173, models/vae_model.py:708-726, test.py:567-569)."""
    F = protein.ca_full.shape[0]
    frames = list(range(F)) if frames is None else list(frames)
    L = protein.L
    z_full = protein.restype_full.to(torch.float32)
    og, cg, nbrs = [], [], []
    for k, f in enumerate(frames):
        full = torch.cat([z_full[:, None], protein.ca_full[f]], dim=1)        # [L+2, 4]
        og.append(full)
        cg.append(full[1:-1])
        nbrs.append(radius_graph(full[1:-1, 1:]) + k * L)
    nf = len(frames)
    return {
        "CG_nxyz": torch.cat(cg, 0),
        "OG_CG_nxyz": torch.cat(og, 0),
        "num_CGs": torch.full((nf,), L, dtype=torch.int64),
        "num_atoms": torch.full((nf,), protein.num_atoms, dtype=torch.int64),
        "CG_nbr_list": torch.cat(nbrs, 0),
        "CG_mapping": torch.zeros(nf * protein.num_atoms, dtype=torch.int64),
        "prot_idx": torch.full((nf,), prot_idx, dtype=torch.int64),
    }


def collate_many(proteins, frame: int = 0) -> dict:
    """One batch dict over several proteins (one frame each), offsets as CG_collate applies them
    (utils/dataset_module.py:259-295: neighbour lists shifted by the running residue count)."""
    parts = [collate(p, [frame], prot_idx=i) for i, p in enumerate(proteins)]
    out, off = {}, 0
    nbrs = []
    for part, p in zip(parts, proteins):
        nbrs.append(part["CG_nbr_list"] + off)
        off += p.L
    for k in parts[0]:
        out[k] = torch.cat(nbrs, 0) if k == "CG_nbr_list" else torch.cat([part[k] for part in parts], 0)
    return out


def latent_noise(shape, seed: int) -> torch.Tensor:
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def eval_loss_case(seed: int, na: int = 3000) -> dict:
    """Seeded inputs of the pair-list losses (shared with the tests): a compact random structure (so that the 1.2 A clash threshold
    is exercised), a noisy copy, bond / neighbour / backbone N-O / interaction pair lists and pi-pi quads."""
    g = torch.Generator().manual_seed(seed)
    xyz = torch.randn(na, 3, generator=g) * 2.5
    recon = xyz + 0.2 * torch.randn(na, 3, generator=g)
    edge = torch.randint(0, na, (5000, 2), generator=g)
    nbr = torch.cat([edge[:1500], edge[100:200].flip(1), torch.randint(0, na, (20000, 2), generator=g)])
    nbr = torch.cat([nbr, nbr[-50:]])
    bb = torch.randint(0, na, (700, 2), generator=g)
    inter = torch.randint(0, na, (400, 2), generator=g)
    pipi = torch.randint(0, na, (37, 4), generator=g)
    return dict(xyz=xyz, recon=recon, edge=edge, nbr=nbr, bb=bb, inter=inter, pipi=pipi)
