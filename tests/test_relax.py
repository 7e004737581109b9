"""CPU tests of the restrained clash relaxation: the float64 restatement (tests/relax_oracle.py) on planted geometry -- its restraint
lists, its forces against central finite differences of its energy, its fixed points -- and the argument checks of Backmapper.relax,
Plan.relax and the `relax=` option of the trajectory methods, which all run before any device call."""
import math

import numpy as np
import pytest
import torch

from codlad_b200 import sampler
from codlad_b200.engine import check_relax_args
from tests import relax_oracle as O
from tests.test_repair import Frame


def _args(fr):
    return fr.slot_atom, fr.out_off, fr.lengths, fr.frame_of, fr.L


def test_restraint_lists_of_a_straight_chain():
    """In Frame's geometry the slots of a residue are 2 A apart on a line, so the intra-residue partners within 3 A are the slot
    neighbours; the peptide partners come at any distance, residue before first, residue after last."""
    fr = Frame(L=6, n=5, NB=2)
    partner, d0 = O.restraint_lists(fr.xyz, *_args(fr))
    assert partner.shape == d0.shape == (2, 6, 14, O.RCAP)
    assert torch.equal(partner[0], partner[1]) and torch.equal(d0[0], d0[1])
    row = lambda i, t: [q for q in partner[0, i, t].tolist() if q >= 0]
    assert row(2, O.SLOT_N) == [14 + O.SLOT_O, 14 + O.SLOT_C, 14 + O.SLOT_CA, 28 + O.SLOT_O, 28 + O.SLOT_C]
    assert row(2, O.SLOT_CA) == [14 + O.SLOT_C, 28 + O.SLOT_C, 28 + 4, 42 + O.SLOT_N]
    assert row(2, O.SLOT_C) == [28 + O.SLOT_N, 28 + O.SLOT_CA, 42 + O.SLOT_N, 42 + O.SLOT_CA]
    assert row(0, O.SLOT_N) == [O.SLOT_O, O.SLOT_C]                 # no residue before the first
    assert row(4, O.SLOT_C) == [56 + O.SLOT_N, 56 + O.SLOT_CA]       # none after the last real residue
    assert row(5, O.SLOT_N) == []                                    # padded
    assert bool((d0[0, 2, O.SLOT_N, 3:5] == d0[0, 2, O.SLOT_N, 3]).all()) and abs(float(d0[0, 2, O.SLOT_N, 3]) - 2.0) < 1e-6
    assert bool((partner[0, :5] >= 0).sum(-1).max() <= O.RCAP)


def test_restraint_capacity_is_reached_by_a_compact_residue():
    """Every slot of residue 2 within 3 A of every other: N has 13 intra-residue partners and the 3 peptide ones, RCAP = 16."""
    fr = Frame(L=4, n=4)
    for t in range(14):
        fr.xyz[fr.row(0, 2, t)] = torch.tensor([20.0 + 0.1 * t, 0.0, 0.0])
    partner, _ = O.restraint_lists(fr.xyz, *_args(fr))
    assert int((partner[0, 2, O.SLOT_N] >= 0).sum()) == 16
    assert int((partner[0, 2, O.SLOT_CA] >= 0).sum()) == 15


def _planted():
    fr = Frame(L=6, n=5, NB=2)
    fr.plant(0, 1, 6, 3, 9, [0.3, 0.2, 0.1])        # two side-chain atoms 0.37 A apart
    fr.plant(0, 0, 5, 2, 0, [0.5, -0.4, 0.2])       # a side-chain atom on an O two residues on
    return fr


def test_forces_match_finite_differences():
    fr = _planted()
    m = O.Member(O.restraint_lists(fr.xyz, *_args(fr)), *_args(fr)[:-1], 0, fr.L)
    x = fr.xyz.double().numpy()[m.rows]
    rng = np.random.default_rng(0)
    x = x + rng.normal(scale=0.05, size=x.shape)    # off the restraints' minimum, so both kinds of term act
    c = O.cutoff(1.2)
    f = m.forces(x, c)
    assert np.abs(f).max() > 1.0
    h = 1e-6
    for k in rng.choice(len(x), 12, replace=False):
        for a in range(3):
            xp, xm = x.copy(), x.copy()
            xp[k, a] += h
            xm[k, a] -= h
            fd = -(m.energy(xp, c) - m.energy(xm, c)) / (2 * h)
            assert abs(fd - f[k, a]) < 1e-5 * max(1.0, abs(f[k, a])), (k, a, fd, f[k, a])


def test_relaxation_separates_the_planted_pairs_and_keeps_the_trace():
    fr = _planted()
    out = O.relax(fr.xyz, *_args(fr), 1.2, sampler.RELAX_ITERATIONS)
    x32 = torch.tensor(out, dtype=torch.float32)
    counts, _ = O.repulsion_counts(x32, *_args(fr), 1.2)
    assert int(counts.sum()) == 0
    ca = [fr.row(b, i, O.SLOT_CA) for b in range(2) for i in range(5)]
    assert np.array_equal(out[ca], fr.xyz.double().numpy()[ca])
    member1 = slice(int(fr.out_off[1]), None)
    assert np.array_equal(out[member1], fr.xyz.double().numpy()[member1])       # nothing under c: the input exactly


def test_no_pair_under_c_returns_the_input_exactly():
    fr = Frame(L=6, n=5, NB=2)
    out = O.relax(fr.xyz, *_args(fr), 2.0, 20)
    assert np.array_equal(out, fr.xyz.double().numpy())


def test_step_cap_and_fixed_atoms():
    fr = _planted()
    m = O.Member(O.restraint_lists(fr.xyz, *_args(fr)), *_args(fr)[:-1], 0, fr.L)
    x = fr.xyz.double().numpy()[m.rows]
    x[5] = np.nan                                    # a non-finite atom: it stays, and its pairs are skipped
    y = m.step(x, O.cutoff(1.2))
    step = np.linalg.norm(y - x, axis=1)
    assert np.isnan(y[5]).all()
    assert np.nanmax(step) <= O.MAX_STEP * (1 + 1e-12) and np.nanmax(step) > 0
    assert np.array_equal(y[m.fixed], x[m.fixed])
    assert np.isfinite(np.delete(y, 5, 0)).all()


# ------------------------------------------------------------------------------------------------ argument checks
@pytest.mark.parametrize("threshold", [0, 0.0, -1.0, 2.0001, 2.5, math.nan, math.inf, True, "1.2", None])
def test_bad_threshold(threshold):
    with pytest.raises(ValueError, match="threshold"):
        check_relax_args(threshold, 10)


@pytest.mark.parametrize("iterations", [-1, 100_001, 1.0, True, None, "5"])
def test_bad_iterations(iterations):
    with pytest.raises(ValueError, match="iterations"):
        check_relax_args(1.2, iterations)


def test_good_arguments():
    for thr, it in ((1.2, 0), (2.0, 100_000), (np.float32(0.5), np.int64(7)), (1e-6, 1)):
        check_relax_args(thr, it)


@pytest.mark.parametrize("relax", [1, [], "yes", {"iters": 5}, {"threshold": 3.0}, {"iterations": -1}, {"iterations": 2.5}])
def test_bad_relax_option(relax):
    with pytest.raises(ValueError):
        sampler.relax_option(relax)


def test_relax_option_defaults():
    assert sampler.relax_option(None) is None
    assert sampler.relax_option({}) == {"iterations": sampler.RELAX_ITERATIONS, "threshold": 1.2}
    assert sampler.relax_option({"threshold": 0.8}) == {"iterations": sampler.RELAX_ITERATIONS, "threshold": 0.8}


class _NoDevice:
    """Stands for a plan / frame set / native call: any use of it is an error, so a refusal must come first."""

    def __getattr__(self, name):
        raise AssertionError(f"touched .{name} before refusing")


def _stub_backmapper():
    bm = object.__new__(sampler.Backmapper)
    bm.T, bm.k_neighbors = 10, 64
    return bm


def test_backmapper_relax_refuses_before_any_device_call():
    bm, nd = _stub_backmapper(), _NoDevice()
    good = {k: nd for k in ("latent", "idx", "zq", "ic_recon", "xyz")}
    for out in (None, {"xyz": nd}, [good]):
        with pytest.raises(ValueError, match="out"):
            bm.relax(nd, nd, out)
    for kw in ({"threshold": 2.5}, {"threshold": 0.0}, {"iterations": -1}, {"iterations": 1.5}):
        with pytest.raises(ValueError):
            bm.relax(nd, nd, good, **kw)


def test_trajectory_relax_options_refuse_before_any_device_call():
    bm = _stub_backmapper()
    ca = torch.zeros(3, 7, 3)
    restype = torch.zeros(7, dtype=torch.int64)
    for bad in ({"threshold": 2.1}, {"steps": 3}, 5):
        with pytest.raises(ValueError):
            bm.backmap_coords(ca, restype, None, relax=bad)
        with pytest.raises(ValueError):
            bm.backmap_trajectory([None] * 3, None, relax=bad)
        sb = sampler.ShardedBackmapper(bm, rank=0, world=1)
        with pytest.raises(ValueError):
            sb.backmap_coords([(ca, restype, None)], relax=bad, _compute=lambda *a, **k: pytest.fail("computed"))
