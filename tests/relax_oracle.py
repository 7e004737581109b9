"""Float64 restatement of the restrained clash relaxation of cb2_plan_relax (Backmapper.relax).

Per member: the restraint set (intra-residue pairs of present atoms within R_RESTRAIN of each other at the input, and the four
peptide pairs C(i)-N(i+1), CA(i)-N(i+1), O(i)-N(i+1), C(i)-CA(i+1)), each held at its input distance d0; the repulsion set
(every pair of atoms of two different residues, the peptide pairs left out, closer than c = threshold + RELAX_MARGIN);
E = sum_R K_S (d - d0)^2 + sum_rep K_R (c - d)^2 with d = sqrt(|x_p - x_q|^2 + 1e-7); and the capped Jacobi update
x += alpha F, scaled to MAX_STEP where longer, for every atom but the C-alphas and non-finite atoms.  The restraint lists and
their d0 are fp32 values, formed as the pinned oracle's `_pd` (the distance of clash_result) forms them but with the kernel's
summation order (x, then y, then z; `_pd`'s torch sum differs from it in the last bit for about 0.6 % of pairs), so they can be
compared bit for bit; the iteration itself runs in float64.
"""
import numpy as np
import torch

from oracle.restate import EVAL_EPS as EPS

SLOTS, SLOT_O, SLOT_N, SLOT_C, SLOT_CA = 14, 0, 1, 2, 3
RCAP = 16
R_RESTRAIN = 3.0
RELAX_MARGIN = 0.2
K_S, K_R, ALPHA, MAX_STEP = 1.0, 10.0, 0.05, 0.1
PEPTIDE = ((SLOT_C, SLOT_N), (SLOT_CA, SLOT_N), (SLOT_O, SLOT_N), (SLOT_C, SLOT_CA))    # (slot in residue i, slot in i + 1)


def pair_dist32(xyz, pairs):
    """_pd with atom_pair_dist's operation order: fp32 differences, squares summed in x, y, z order from 0, then 1e-7, then a
    correctly rounded sqrt."""
    x = torch.as_tensor(xyz, dtype=torch.float32).cpu().numpy()
    p = torch.as_tensor(pairs).long().cpu().numpy()
    d = x[p[:, 0]] - x[p[:, 1]]
    s = np.float32(0) + d[:, 0] * d[:, 0]
    s = s + d[:, 1] * d[:, 1]
    s = s + d[:, 2] * d[:, 2]
    with np.errstate(invalid="ignore"):
        return torch.from_numpy(np.sqrt(s + np.float32(EPS)))


def cutoff(threshold):
    """c = threshold + RELAX_MARGIN, rounded to fp32 as the kernel forms it."""
    return float(np.float32(threshold) + np.float32(RELAX_MARGIN))


def _member(slot_atom, out_off, lengths, frame_of, b, L):
    """(slot-grid table sa [n, 14] of member b's output rows, -1 where absent; n = its length)."""
    f = int(frame_of[b])
    n = int(lengths[f])
    sa = torch.as_tensor(slot_atom[f]).reshape(L, SLOTS)[:n].long().clone()
    sa[sa >= 0] += int(out_off[b])
    return sa, n


def _candidates(t):
    """The partners atom slot t may be restrained to, in list order: (residue offset, slot, peptide pair?)."""
    return ([(-1, u, True) for u in range(SLOTS) if (u, t) in PEPTIDE] + [(0, u, False) for u in range(SLOTS) if u != t]
            + [(1, u, True) for u in range(SLOTS) if (t, u) in PEPTIDE])


def restraint_lists(xyz, slot_atom, out_off, lengths, frame_of, L):
    """partner int32 [NB, L, 14, RCAP] (member-local slot index j * 14 + u, -1 past the end) and d0 float32 (0 past the end): per
    atom, its restrained partners in the order residue ascending, then slot ascending, with d0 = _pd at the input.  Pairs whose d0 is
    not finite are left out."""
    xyz = torch.as_tensor(xyz, dtype=torch.float32).cpu()
    NB = int(torch.as_tensor(frame_of).numel())
    partner = torch.full((NB, L, SLOTS, RCAP), -1, dtype=torch.int32)
    d0 = torch.zeros(NB, L, SLOTS, RCAP, dtype=torch.float32)
    for b in range(NB):
        sa, n = _member(slot_atom, out_off, lengths, frame_of, b, L)
        pad = torch.full((n + 2, SLOTS), -1, dtype=torch.long)
        pad[1:-1] = sa                                   # residues -1 and n are absent
        i = torch.arange(n)
        for t in range(SLOTS):
            cand = _candidates(t)
            j = i[:, None] + torch.tensor([dj for dj, _, _ in cand])[None]             # [n, C]
            u = torch.tensor([u for _, u, _ in cand]).expand(n, -1)
            pep = torch.tensor([p for _, _, p in cand]).expand(n, -1)
            p_row, q_row = sa[:, t, None].expand(-1, len(cand)), pad[j + 1, u]
            ok = (p_row >= 0) & (q_row >= 0)
            d = torch.full(ok.shape, float("nan"))
            d[ok] = pair_dist32(xyz, torch.stack((p_row[ok], q_row[ok]), 1))
            keep = ok & torch.isfinite(d) & (pep | (d <= R_RESTRAIN))
            k = torch.cumsum(keep.long(), 1) - 1
            ii, cc = torch.nonzero(keep, as_tuple=True)
            partner[b, ii, t, k[ii, cc]] = (j[ii, cc] * SLOTS + u[ii, cc]).to(torch.int32)
            d0[b, ii, t, k[ii, cc]] = d[ii, cc]
    return partner, d0


def _peptide_mask(res, slot):
    """[P, P] bool: (p, q) is a peptide pair, seen from either side."""
    a = np.zeros((len(res), len(res)), dtype=bool)
    for s, u in PEPTIDE:
        a |= (res[:, None] + 1 == res[None, :]) & (slot[:, None] == s) & (slot[None, :] == u)
    return a | a.T


class Member:
    """One member's atoms (rows of the output xyz), their restraints and the masks the energy needs."""

    def __init__(self, lists, slot_atom, out_off, lengths, frame_of, b, L):
        sa, n = _member(slot_atom, out_off, lengths, frame_of, b, L)
        res, slot = np.nonzero(sa.numpy() >= 0)
        self.rows = sa.numpy()[res, slot]
        self.res, self.slot = res, slot
        index = {(int(r), int(s)): k for k, (r, s) in enumerate(zip(res, slot))}
        partner, d0 = lists
        P = len(self.rows)
        self.rest = np.zeros((P, P), dtype=bool)
        self.d0 = np.zeros((P, P))
        for k, (r, s) in enumerate(zip(res, slot)):
            for q, d in zip(partner[b, r, s].tolist(), d0[b, r, s].tolist()):
                if q >= 0:
                    kk = index[(q // SLOTS, q % SLOTS)]
                    self.rest[k, kk], self.d0[k, kk] = True, d
        self.inter = (res[:, None] != res[None, :]) & ~_peptide_mask(res, slot)
        self.fixed = slot == SLOT_CA

    def terms(self, x, c):
        """(diff [P, P, 3], d [P, P], finite pair mask [P, P], repulsion mask [P, P]) at positions x [P, 3] float64."""
        diff = x[:, None, :] - x[None, :, :]
        with np.errstate(invalid="ignore"):
            d = np.sqrt((diff * diff).sum(-1) + EPS)
            ok = np.isfinite(x).all(1)
            fin = ok[:, None] & ok[None, :]
            rep = self.inter & fin & (d < c)
        return diff, d, fin, rep

    def energy(self, x, c):
        diff, d, fin, rep = self.terms(x, c)
        rest = self.rest & fin
        return 0.5 * (K_S * ((d - self.d0) ** 2)[rest].sum() + K_R * ((c - d) ** 2)[rep].sum())    # every pair is listed twice

    def forces(self, x, c):
        diff, d, fin, rep = self.terms(x, c)
        rest = self.rest & fin
        g = np.zeros_like(d)
        g[rest] = -2 * K_S * (d - self.d0)[rest] / d[rest]
        g[rep] += 2 * K_R * (c - d)[rep] / d[rep]
        return (g[..., None] * np.where(fin[..., None], diff, 0.0)).sum(1)

    def step(self, x, c):
        f = self.forces(x, c)
        dx = ALPHA * f
        n = np.linalg.norm(dx, axis=1)
        scale = np.where(n > MAX_STEP, MAX_STEP / np.where(n > 0, n, 1.0), 1.0)
        dx = dx * scale[:, None]
        move = ~self.fixed & np.isfinite(x).all(1)
        return np.where(move[:, None], x + dx, x)


def relax(xyz, slot_atom, out_off, lengths, frame_of, L, threshold, iterations):
    """The relaxed coordinates (float64 [total atoms, 3]): rows of absent slots and padded residues as given."""
    xyz32 = torch.as_tensor(xyz, dtype=torch.float32).cpu()
    out = xyz32.double().numpy().copy()
    c = cutoff(threshold)
    lists = restraint_lists(xyz32, slot_atom, out_off, lengths, frame_of, L)
    for b in range(int(torch.as_tensor(frame_of).numel())):
        m = Member(lists, slot_atom, out_off, lengths, frame_of, b, L)
        x = out[m.rows]
        if not m.inter.any() or not m.terms(x, c)[3].any():
            continue                     # no pair under c: the input exactly (the energy's minimum)
        for _ in range(iterations):
            x = m.step(x, c)
        out[m.rows] = x
    return out


def repulsion_counts(xyz, slot_atom, out_off, lengths, frame_of, L, c):
    """int32 [NB, L, 14]: per atom, the inter-residue non-peptide partners closer than c by pair_dist32 (the kernel's distance),
    and the smallest |d - c| over all such pairs of every member (to check that no pair sits at the cutoff's rounding edge)."""
    xyz = torch.as_tensor(xyz, dtype=torch.float32).cpu()
    NB = int(torch.as_tensor(frame_of).numel())
    counts = torch.zeros(NB, L, SLOTS, dtype=torch.int32)
    gap = float("inf")
    for b in range(NB):
        sa, n = _member(slot_atom, out_off, lengths, frame_of, b, L)
        res, slot = np.nonzero(sa.numpy() >= 0)
        rows = torch.as_tensor(sa.numpy()[res, slot])
        P = len(rows)
        p, q = torch.meshgrid(torch.arange(P), torch.arange(P), indexing="ij")
        d = pair_dist32(xyz, torch.stack((rows[p.reshape(-1)], rows[q.reshape(-1)]), 1)).view(P, P)
        inter = torch.as_tensor((res[:, None] != res[None, :]) & ~_peptide_mask(res, slot))
        hit = inter & (d < c)
        counts[b, res, slot] = hit.sum(1).to(torch.int32)
        if inter.any():
            gap = min(gap, float((d[inter].double() - c).abs().min()))
    return counts, gap
