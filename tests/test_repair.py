"""CPU tests of clash-driven repair: the brute-force clash oracle (tests/clash_oracle.py) on planted geometry with hand-counted
answers, its keep mask, the acceptance rule of Backmapper.repair and the argument checks that run before any device call."""
import math

import numpy as np
import pytest
import torch

from codlad_b200.engine import check_clash_args
from codlad_b200.sampler import clash_pair_totals, repair_accept
from oracle.restate import _pd
from tests import clash_oracle as O

THR = 1.2


def _edge_offsets(thr=THR):
    """(inside, outside): the two adjacent fp32 offsets along x around the threshold, for an atom at the origin."""
    d = np.float32(thr)
    dist = lambda x: float(_pd(torch.tensor([[0.0, 0.0, 0.0], [float(x), 0.0, 0.0]]), torch.tensor([[0, 1]]))[0])
    while dist(d) >= thr:
        d = np.nextafter(d, np.float32(0))
    return float(d), float(np.nextafter(d, np.float32(2 * thr)))


class Frame:
    """One frame of L residues (the first n real) and NB members on it; slot t of residue i of member b sits at (10 i, 100 b, 2 t),
    so that nothing clashes until an atom is planted."""

    def __init__(self, L=6, n=5, NB=1, absent=()):
        self.L, self.n, self.NB = L, n, NB
        sa = torch.full((L, 14), -1, dtype=torch.int32)
        k = 0
        for i in range(n):
            for t in range(14):
                if (i, t) not in absent:
                    sa[i, t] = k
                    k += 1
        self.na = k
        self.slot_atom = sa.reshape(1, L * 14)
        self.lengths = torch.tensor([n], dtype=torch.int32)
        self.frame_of = torch.zeros(NB, dtype=torch.int32)
        self.out_off = torch.arange(NB, dtype=torch.int64) * k
        self.xyz = torch.zeros(NB * k, 3)
        for b in range(NB):
            for i in range(n):
                for t in range(14):
                    if sa[i, t] >= 0:
                        self.xyz[self.row(b, i, t)] = torch.tensor([10.0 * i, 100.0 * b, 2.0 * t])

    def row(self, b, i, t):
        return int(self.out_off[b]) + int(self.slot_atom[0, i * 14 + t])

    def plant(self, b, i, t, j, u, offset):
        """Put atom (j, u) of member b at atom (i, t) + offset."""
        self.xyz[self.row(b, j, u)] = self.xyz[self.row(b, i, t)] + torch.tensor(offset, dtype=torch.float32)

    def counts(self, thr=THR):
        return O.residue_clashes(self.xyz, self.slot_atom, self.out_off, self.lengths, self.frame_of, self.L, thr)


def test_unplanted_frame_has_no_clash():
    assert int(Frame(NB=2).counts().sum()) == 0


def test_threshold_edge():
    inside, outside = _edge_offsets()
    assert inside < outside
    for off, want in ((inside, 1), (outside, 0)):
        fr = Frame()
        fr.xyz[fr.row(0, 3, 6)] = fr.xyz[fr.row(0, 0, 5)] + torch.tensor([off, 0.0, 0.0])
        c = fr.counts()
        assert c[0, 0] == want and c[0, 3] == want and int(c.sum()) == 2 * want


def test_peptide_pair_is_excluded_but_not_its_neighbours():
    fr = Frame()
    fr.plant(0, 1, 2, 2, 1, [0.5, 0.0, 0.0])      # C(1)-N(2): the peptide bond, not a clash
    assert int(fr.counts().sum()) == 0
    fr = Frame()
    fr.plant(0, 1, 2, 3, 1, [0.5, 0.0, 0.0])      # C(1)-N(3): a clash
    assert fr.counts()[0].tolist() == [0, 1, 0, 1, 0, 0]
    fr = Frame()
    fr.plant(0, 1, 1, 2, 2, [0.5, 0.0, 0.0])      # N(1)-C(2) is not the peptide pair either
    assert fr.counts()[0].tolist() == [0, 1, 1, 0, 0, 0]
    fr = Frame()
    fr.plant(0, 1, 0, 2, 1, [0.5, 0.0, 0.0])      # O(1)-N(2): neighbours in sequence, other atoms
    assert fr.counts()[0].tolist() == [0, 1, 1, 0, 0, 0]


def test_one_atom_near_several():
    """An atom within the threshold of three atoms of another residue counts three pairs for each side."""
    fr = Frame()
    for t in (4, 5, 6):
        fr.xyz[fr.row(0, 4, t)] = torch.tensor([5.0 + 0.1 * t, 50.0, 50.0])
    fr.xyz[fr.row(0, 0, 3)] = torch.tensor([5.5, 50.3, 50.0])
    c = fr.counts()
    assert c[0].tolist() == [3, 0, 0, 0, 3, 0]


def test_absent_slots():
    """Absent slots are no atoms: a residue with only its backbone clashes through the atoms it has."""
    fr = Frame(absent={(2, t) for t in range(4, 14)} | {(3, 1)})
    fr.plant(0, 2, 3, 0, 7, [0.3, 0.0, 0.0])
    fr.plant(0, 2, 2, 3, 0, [0.0, 0.4, 0.0])      # C(2)-O(3): counted (N(3) is absent, O is not N)
    assert fr.counts()[0].tolist() == [1, 0, 2, 1, 0, 0]


def test_padded_residues_and_several_members():
    """Padded rows count nothing and keep True; members of one frame are independent even where their atoms coincide."""
    fr = Frame(L=6, n=4, NB=3)
    fr.xyz[fr.out_off[1]:fr.out_off[2]] = fr.xyz[:fr.out_off[1]]     # member 1 on top of member 0
    fr.plant(0, 0, 4, 3, 9, [0.2, 0.2, 0.2])
    fr.plant(2, 1, 5, 3, 5, [0.0, 0.0, 0.7])
    fr.plant(2, 1, 6, 3, 6, [0.0, 0.0, 0.7])
    c = fr.counts()
    assert c.tolist() == [[1, 0, 0, 1, 0, 0], [0] * 6, [0, 2, 0, 2, 0, 0]]
    nbr = torch.tensor([sorted(range(6), key=lambda j: (abs(j - i), j)) for i in range(6)])[None]
    keep = O.keep_mask(c, nbr, fr.lengths, fr.frame_of, 0)
    assert keep.tolist() == [[False, True, True, False, True, True], [True] * 6, [True, False, True, False, True, True]]


def test_keep_mask_grow():
    """grow counts the nearest other residues: the residue itself is skipped wherever it is in its row."""
    counts = torch.tensor([[0, 0, 0, 2, 0, 0, 0, 0]], dtype=torch.int32)
    lengths, frame_of = torch.tensor([7]), torch.tensor([0])
    nbr = torch.tensor([sorted(range(8), key=lambda j: (abs(j - i), j)) for i in range(8)])[None]
    nbr[0, 4, :2] = torch.tensor([3, 4])          # a tie that puts another residue before the residue itself
    row = lambda g: O.keep_mask(counts, nbr, lengths, frame_of, g)[0].tolist()
    assert row(0) == [True, True, True, False, True, True, True, True]
    assert row(1) == [True, True, True, False, False, True, True, True]        # 4: entry 0 is residue 3
    assert row(2) == [True, True, False, False, False, True, True, True]       # 2: entries 1, 3
    assert row(3) == [False, False, False, False, False, False, True, True]    # 6: entries 5, 7, 4; 7 is padded: always True


def test_acceptance_rule_and_pair_totals():
    counts = torch.tensor([[1, 0, 1, 0], [0, 0, 0, 0], [3, 1, 2, 0]], dtype=torch.int32)
    assert clash_pair_totals(counts).tolist() == [1, 0, 3]
    assert clash_pair_totals(counts).dtype == torch.int64
    prev, new = torch.tensor([3, 0, 2, 5]), torch.tensor([1, 0, 2, 6])
    assert repair_accept(prev, new).tolist() == [True, False, False, False]


@pytest.mark.parametrize("threshold", [0, 0.0, -1.2, math.nan, math.inf, -math.inf, True, "1.2", None])
def test_bad_threshold(threshold):
    with pytest.raises(ValueError, match="threshold"):
        check_clash_args(threshold, 0, 64)


@pytest.mark.parametrize("grow", [-1, 64, 65, 1.0, True, None])
def test_bad_grow(grow):
    with pytest.raises(ValueError, match="grow"):
        check_clash_args(1.2, grow, 64)


def test_good_arguments():
    for thr, grow, K in ((1.2, 0, 64), (np.float32(2.5), 63, 64), (3, np.int64(7), 48), (0.5, 0, 0)):
        check_clash_args(thr, grow, K)
    with pytest.raises(ValueError):
        check_clash_args(1.2, 1, 0)
