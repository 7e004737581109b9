"""CPU restatement of the per-residue clash counts and keep mask of cb2_plan_residue_clashes (Backmapper.residue_clashes).

Brute force: every atom pair of two different residues of a member, the peptide pair C(i)-N(i+1) left out, d from the pinned
oracle's `_pd` (the distance of clash_result, test.py:118-139) and `d < threshold`.  The reference has no per-residue form of
the criterion, so this is unpinned; it is tied to clash_result through `_pd`, and the GPU tests tie it to cb2_pair_losses.
"""
import torch

from oracle.restate import _pd

SLOTS, SLOT_N, SLOT_C = 14, 1, 2


def member_pairs(slot_atom, out_off, lengths, frame_of, b, L):
    """All ordered atom pairs (a, c) of member b with a and c in different residues, the peptide pair left out.
    Returns (pairs [P, 2] int64 atom rows, residue of a [P], number of residues n)."""
    f = int(frame_of[b])
    n = int(lengths[f])
    sa = torch.as_tensor(slot_atom[f]).reshape(L, SLOTS)[:n].long()
    res = torch.arange(n)[:, None].expand(n, SLOTS)
    slot = torch.arange(SLOTS)[None].expand(n, SLOTS)
    present = sa >= 0
    atom, r, s = sa[present] + int(out_off[b]), res[present], slot[present]
    p, q = torch.meshgrid(torch.arange(atom.numel()), torch.arange(atom.numel()), indexing="ij")
    p, q = p.reshape(-1), q.reshape(-1)
    peptide = ((r[q] == r[p] + 1) & (s[p] == SLOT_C) & (s[q] == SLOT_N)) | ((r[q] == r[p] - 1) & (s[p] == SLOT_N) & (s[q] == SLOT_C))
    sel = (r[p] != r[q]) & ~peptide
    return torch.stack((atom[p[sel]], atom[q[sel]]), 1), r[p[sel]], n


def residue_clashes(xyz, slot_atom, out_off, lengths, frame_of, L, threshold):
    """counts [NB, L] int32: per residue, the atom pairs with other residues of its member closer than `threshold`."""
    xyz = torch.as_tensor(xyz, dtype=torch.float32).cpu()
    NB = int(torch.as_tensor(frame_of).numel())
    counts = torch.zeros(NB, L, dtype=torch.int32)
    for b in range(NB):
        pairs, r, n = member_pairs(slot_atom, out_off, lengths, frame_of, b, L)
        if pairs.numel():
            hit = _pd(xyz, pairs) < threshold
            counts[b, :n] = torch.bincount(r[hit], minlength=n).to(torch.int32)
    return counts


def unordered_pairs(slot_atom, out_off, lengths, frame_of, b, L):
    """The inter-residue, non-peptide atom pairs of member b once each (a < c): the pair list of cb2_pair_losses."""
    pairs, _, _ = member_pairs(slot_atom, out_off, lengths, frame_of, b, L)
    return pairs[pairs[:, 0] < pairs[:, 1]]


def keep_mask(counts, nbr_idx, lengths, frame_of, grow):
    """keep [NB, L] bool: False where residue i or one of its first `grow` entries of nbr_idx [F, L, K] other than itself has a
    clash; True elsewhere and on padded rows."""
    NB, L = counts.shape
    keep = torch.ones(NB, L, dtype=torch.bool)
    for b in range(NB):
        f = int(frame_of[b])
        for i in range(int(lengths[f])):
            bad, taken = bool(counts[b, i] > 0), 0
            for j in torch.as_tensor(nbr_idx[f, i]).tolist():
                if bad or taken >= grow:
                    break
                if j == i:
                    continue
                taken += 1
                bad = bool(counts[b, j] > 0)
            keep[b, i] = not bad
    return keep
