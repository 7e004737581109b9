"""CPU tests of partial-noise refinement and warm-started trajectory backmapping: the oracle's restatement (tests/refine_oracle.py)
tied to the pinned DDPM oracle and to the DDIM oracle (steps = T, no kept row: the plain loop from the level-T start), every row
kept, the argument checks that run before any device call, the chunk split of backmap_trajectory and the residue gather of
residue_motion."""
import numpy as np
import pytest
import torch

from codlad_b200 import synthetic, topology, weights
from codlad_b200.engine import check_start_steps
from codlad_b200.sampler import Backmapper, frames_from_batch, residue_atom_ranges, trajectory_chunks
from oracle import restate as R
from tests import ddim_oracle as D
from tests import inpaint_oracle as I
from tests import refine_oracle as O


@pytest.fixture
def one_thread():
    """The identities below compare two CPU loops bit for bit; a matrix product may sum in another order when the library picks
    another thread count between calls, so both loops run on one thread."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _case(L=24, B=2, seed=91):
    prot = synthetic.make_protein(L, 1, seed=seed)
    X = prot.ca_full[:, 1:-1].expand(B, -1, -1).contiguous()
    cg_z = prot.restype_full[1:-1][None].expand(B, -1).contiguous()
    mask = torch.ones(B, L, dtype=torch.bool)
    mask[1, L - 5:] = False                                             # a padded tail on the second member
    return dict(sd=weights.init_denoiser_state(0), X=X, cg_z=cg_z, mask=mask, z=synthetic.latent_noise((B, L, 3), seed + 1),
                noises=synthetic.latent_noise((10, B, L, 3), seed + 2), x0=synthetic.latent_noise((B, L, 3), seed + 3))


def _level(spacing, r, x0, z):
    q = I.level_table(spacing)
    return q[r, 0] * x0 + q[r, 1] * z


def test_full_start_without_kept_rows_is_the_plain_ddpm_loop(one_thread):
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    got = O.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], c["noises"], "10", 10, keep, c["x0"], "ddpm")
    want = R.sample_loop(c["sd"], _level("10", 10, c["x0"], c["z"]), c["X"], c["cg_z"], c["mask"], c["noises"], R.respaced_schedule(10))
    assert torch.equal(got, want)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_full_start_without_kept_rows_is_the_plain_ddim_loop(one_thread, eta):
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    noises = c["noises"] if eta != 0 else None
    got = O.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], noises, "10", 10, keep, c["x0"], "ddim", eta)
    want = D.sample_loop(c["sd"], _level("10", 10, c["x0"], c["z"]), c["X"], c["cg_z"], c["mask"], noises, D.schedule("10"), eta)
    assert torch.equal(got, want)


def test_level_start_is_fp32_without_fma():
    """The start row of every member is two rounded fp32 products and one rounded sum of the float64-rounded level."""
    c = _case()
    q = I.level_table("10").numpy()
    got = _level("10", 4, c["x0"], c["z"]).numpy()
    x0, z = c["x0"].numpy(), c["z"].numpy()
    want = (np.float32(q[4, 0]) * x0).astype(np.float32) + (np.float32(q[4, 1]) * z).astype(np.float32)
    assert got.dtype == np.float32 and np.array_equal(got, want)


@pytest.mark.parametrize("sampler,eta,steps", [("ddpm", 0.0, 1), ("ddpm", 0.0, 5), ("ddim", 0.0, 5), ("ddim", 1.0, 10)])
def test_every_row_kept_returns_x0(sampler, eta, steps):
    c = _case()
    keep = torch.ones(c["mask"].shape, dtype=torch.bool)
    noises = c["noises"] if sampler == "ddpm" or eta != 0 else None
    got = O.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], noises, "10", steps, keep, c["x0"], sampler, eta)
    assert torch.equal(got, c["x0"])


def test_short_start_stays_near_x0_and_kept_rows_are_exact():
    """One DDIM step at eta = 0 from the lowest level moves free rows a little; kept rows end at x0 exactly."""
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    keep[:, 3:9] = True
    got = O.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], None, "10", 1, keep, c["x0"], "ddim", 0.0)
    assert torch.equal(got[keep], c["x0"][keep])
    free = ~keep
    assert not torch.equal(got[free], c["x0"][free])


# ---- argument checks (no device is touched) -------------------------------------------------------------------------------------
def _bm(T=10):
    bm = object.__new__(Backmapper)          # the checks below run before any use of the engines
    bm.T = T
    return bm


def _fs(L=12, NB=2):
    prot = synthetic.make_protein(L, 1, seed=5)
    return frames_from_batch(synthetic.collate(prot), prot.info, NB)


@pytest.mark.parametrize("steps", [-1, True, 1.0, "2", None])
def test_set_start_rejects(steps):
    with pytest.raises(ValueError):
        check_start_steps(steps)


@pytest.mark.parametrize("steps", [0, 1, 100])
def test_set_start_accepts(steps):
    check_start_steps(steps)


@pytest.mark.parametrize("steps", [0, 11, -1, True, 2.0, None])
def test_refine_rejects_steps(steps):
    fs = _fs()
    plan = type("P", (), {"device": torch.device("cpu")})()
    with pytest.raises(ValueError, match="steps"):
        _bm().refine(plan, fs, torch.zeros(fs.NB, fs.L, 3), steps)


def test_refine_rejects_latent_and_keep():
    fs = _fs()
    plan = type("P", (), {"device": torch.device("cpu")})()
    lat, keep = torch.zeros(fs.NB, fs.L, 3), torch.zeros(fs.NB, fs.L, dtype=torch.bool)
    for bad_lat, bad_keep in ((lat.double(), keep), (lat[:, :5], keep), (lat[..., :2], keep), (lat, keep.to(torch.uint8)),
                              (lat, keep[:, :5])):
        with pytest.raises(ValueError):
            _bm().refine(plan, fs, bad_lat, 3, keep=bad_keep)


def _trajectory_batches(n=4, L=12):
    prot = synthetic.trajectory(L, n, seed=3)
    return [synthetic.collate(prot, [f]) for f in range(n)], prot.info


@pytest.mark.parametrize("kw", [dict(num_ensemble=0), dict(num_ensemble=True), dict(steps=0), dict(steps=11), dict(steps=1.5),
                                dict(chunks=0), dict(chunks=5), dict(chunks=2.0), dict(chunks=True)])
def test_backmap_trajectory_rejects(kw):
    batches, info = _trajectory_batches()
    with pytest.raises(ValueError):
        _bm().backmap_trajectory(batches, info, **kw)


def test_backmap_trajectory_rejects_mixed_frames():
    batches, info = _trajectory_batches()
    other = synthetic.make_protein(13, 1, seed=4)
    with pytest.raises(ValueError, match="same length"):
        _bm().backmap_trajectory(batches + [synthetic.collate(other)], info)
    prot = synthetic.trajectory(12, 2, seed=3)
    with pytest.raises(ValueError, match="one frame"):
        _bm().backmap_trajectory(batches + [synthetic.collate(prot)], info)


# ---- chunk split ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,chunks,want", [(7, 1, [(0, 7)]), (7, 3, [(0, 3), (3, 2), (5, 2)]), (8, 3, [(0, 3), (3, 3), (6, 2)]),
                                           (6, 3, [(0, 2), (2, 2), (4, 2)]), (5, 5, [(0, 1), (1, 1), (2, 1), (3, 1), (4, 1)]),
                                           (32, 4, [(0, 8), (8, 8), (16, 8), (24, 8)])])
def test_trajectory_chunks(n, chunks, want):
    assert trajectory_chunks(n, chunks) == want


@pytest.mark.parametrize("n", range(1, 30))
def test_trajectory_chunks_cover_the_frames_in_order(n):
    for chunks in range(1, n + 1):
        runs = trajectory_chunks(n, chunks)
        lengths = [k for _, k in runs]
        assert len(runs) == chunks and max(lengths) - min(lengths) <= 1 and min(lengths) >= 1
        assert [f for s, k in runs for f in range(s, s + k)] == list(range(n))
        assert lengths == sorted(lengths, reverse=True)
    with pytest.raises(ValueError, match="exceeds"):
        trajectory_chunks(n, n + 1)


# ---- residue gather of residue_motion ---------------------------------------------------------------------------------------------
def test_residue_atom_ranges():
    """Two proteins of 9 and 6 residues padded to 9, two members on each: every real residue's atoms form one contiguous range
    in slot order at the member's offset, padded rows are left out and every output atom is gathered exactly once."""
    p1, p2 = synthetic.make_protein(9, 1, seed=21), synthetic.make_protein(6, 1, seed=22)
    fs = frames_from_batch(synthetic.collate_many([p1, p2]), [p1.info, p2.info], frame_of=[0, 1, 1, 0])
    atoms, counts, rows = residue_atom_ranges(fs)
    assert atoms.dtype == counts.dtype == rows.dtype == torch.int64
    assert int(counts.sum()) == atoms.numel() == fs.total_atoms
    assert torch.equal(torch.sort(atoms).values, torch.arange(fs.total_atoms))
    restypes = [p1.restype_full[1:-1], p2.restype_full[1:-1]]
    want_rows, o = [], 0
    for b, f in enumerate([0, 1, 1, 0]):
        n = [9, 6][f]
        for i in range(n):
            want_rows.append(b * fs.L + i)
            k = int(topology.ATOM_COUNT[restypes[f][i]])
            r = len(want_rows) - 1
            assert int(counts[r]) == k
            seg = atoms[o:o + k]
            assert torch.equal(seg, seg[0] + torch.arange(k))                       # contiguous in the decoded layout
            slots = fs.slot_atom[f, i * 14:(i + 1) * 14]
            assert torch.equal(seg, int(fs.out_off[b]) + slots[slots >= 0].long())
            o += k
    assert rows.tolist() == want_rows                                             # rows 6..8 of members 1 and 2 are padding
