"""GPU tests of the restrained clash relaxation (run on the B200 box: pytest -m gpu): cb2_plan_relax against the float64 restatement
(tests/relax_oracle.py) -- restraint lists bit for bit, the repulsive pairs evaluated at every iteration against a brute-force pass,
positions after 1 and 20 iterations -- on the decoded samples of test_gpu_repair.py (golden 64 x 1, ragged 80/70 x 4, both tiers)
with planted clashes; the invariants of a default relax; determinism and batch invariance; the trajectory option; and pairs
planted at the repulsion distance and one fp32 step either side of it."""
import numpy as np
import pytest
import torch

from codlad_b200 import sampler, synthetic
from tests import clash_oracle as CO
from tests import relax_oracle as O
from tests.test_gpu_repair import _decoded, _edge_point, states  # noqa: F401  (states is a fixture)

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

THR = 1.2
POS_TOL = {1: 1e-5, 20: 1e-2}       # A, largest coordinate difference from the float64 restatement (measured: 5e-6 / 3.8e-3)


def _args(fs):
    return fs.slot_atom, fs.out_off, fs.lengths, fs.frame_of, fs.L


def _row(fs, b, i, t):
    return int(fs.out_off[b]) + int(fs.slot_atom[int(fs.frame_of[b]), i * 14 + t])


def _last(fs, b, i):
    return int(fs.out_off[b]) + int(fs.slot_atom[int(fs.frame_of[b]), i * 14:(i + 1) * 14].max())


def _planted(fs, xyz):
    """Side-chain atoms put 0.4-1.1 A from an O of another residue, one near in sequence (i + 3) and one far, per member.
    Returns (xyz, planted atom rows)."""
    xyz = xyz.cpu().clone()
    rows = []
    for b in range(fs.NB):
        f = int(fs.frame_of[b])
        n = int(fs.lengths[f])
        side = [r for r in range(n) if int(fs.slot_atom[f, r * 14 + 4]) >= 0]
        for k, (i, j) in enumerate(((side[1 + b], side[1 + b] + 3), (side[-2 - b], side[b]))):
            off = torch.tensor([0.4 + 0.7 * ((b + k) % 3) / 2, 0.0, 0.0])
            xyz[_last(fs, b, i)] = xyz[_row(fs, b, j, O.SLOT_O)] + off
            rows.append(_last(fs, b, i))
    return xyz.cuda(), rows


def _case(states, case, precision):
    bm, plan, fs, out = _decoded(states, case, precision)
    xyz, rows = _planted(fs, out["xyz"])
    return bm, plan, fs, out, xyz, rows


CASES = [(c, p) for c in ("golden", "ragged") for p in ("fp32", "f16")]


@pytest.mark.parametrize("case,precision", CASES)
def test_restraints_and_repulsion_sets_vs_oracle(states, case, precision):
    bm, plan, fs, out, xyz, _ = _case(states, case, precision)
    plan.relax(xyz, THR, 0)
    partner, d0 = O.restraint_lists(xyz.cpu(), *_args(fs))
    assert torch.equal(plan.buffer("relax_partner").cpu(), partner)
    assert torch.equal(plan.buffer("relax_d0").cpu(), d0)
    # the pairs evaluated at iteration t (relax_nrep after t + 1 iterations) against a brute-force pass over x_t (the output of t
    # iterations) with the kernel's own fp32 distance, so pairs at c itself must agree too; across the candidate rebuilds (every 5)
    c = O.cutoff(THR)
    moving = torch.zeros(fs.NB, fs.L, 14, dtype=torch.bool)
    for b in range(fs.NB):
        f = int(fs.frame_of[b])
        sa = fs.slot_atom[f].view(fs.L, 14)
        moving[b, :int(fs.lengths[f])] = sa[:int(fs.lengths[f])] >= 0
    moving[..., O.SLOT_CA] = False
    evaluated = 0
    for t in (0, 1, 4, 5, 9, 10, 14, 19):
        xt, _, _ = plan.relax(xyz, THR, t)
        plan.relax(xyz, THR, t + 1)
        got = plan.buffer("relax_nrep").cpu()
        want, gap = O.repulsion_counts(xt.cpu(), *_args(fs), c)     # gap: repelled pairs settle at c itself, the force's zero
        assert torch.equal(got[moving], want[moving]), t
        assert int(got[~moving].abs().sum()) == 0
        evaluated += int(want[moving].sum())
    assert evaluated > 0
    print(f"{case}/{precision}: repulsive pair evaluations checked {evaluated}")


@pytest.mark.parametrize("case,precision", CASES)
def test_positions_vs_oracle(states, case, precision):
    bm, plan, fs, out, xyz, _ = _case(states, case, precision)
    for it, tol in POS_TOL.items():
        got, _, _ = plan.relax(xyz, THR, it)
        want = O.relax(xyz.cpu(), *_args(fs), THR, it)
        err = float(np.nanmax(np.abs(got.cpu().double().numpy() - want)))
        moved = float(np.nanmax(np.abs(want - xyz.cpu().double().numpy())))
        print(f"{case}/{precision}: {it} iterations, largest difference {err:.2e} A (largest motion {moved:.3f} A)")
        assert err < tol


@pytest.mark.parametrize("case,precision", CASES)
def test_default_relax_invariants(states, case, precision):
    bm, plan, fs, out, xyz, rows = _case(states, case, precision)
    res = bm.relax(plan, fs, dict(out, xyz=xyz))
    new = res["xyz"]
    assert new.shape == xyz.shape and res["clash_pairs"].shape == (2, fs.NB) and res["clash_pairs"].dtype == torch.int64
    for k in ("latent", "idx", "zq", "ic_recon"):
        assert res[k] is out[k]
    # every planted clash is cleared; what is left are pairs the restrained geometry holds together (a C-alpha of the trace, which
    # never moves, or backbone atoms of neighbouring residues), a small share of the random-init decoder's clashes
    counts = CO.residue_clashes(new.cpu(), *_args(fs)[:-1], fs.L, THR)
    assert torch.equal(res["clashes"].cpu(), counts)
    left = []
    for b in range(fs.NB):
        pairs, _, _ = CO.member_pairs(*_args(fs)[:-1], b, fs.L)
        hit = pairs[O.pair_dist32(new.cpu(), pairs) < THR]
        left += [(int(p), int(q)) for p, q in hit.tolist()]
    ca_rows = {_row(fs, b, i, O.SLOT_CA) for b in range(fs.NB) for i in range(int(fs.lengths[int(fs.frame_of[b])]))}
    print(f"{case}/{precision}: clash pairs before / after {res['clash_pairs'].tolist()}, max shift {res['max_shift'].tolist()}, "
          f"max restraint deviation {res['max_restraint_dev'].tolist()}")
    before, after = res["clash_pairs"].sum(1).tolist()
    assert after <= 0.1 * before
    assert not any(p in rows or q in rows for p, q in left), "a planted clash is left"
    # C-alpha rows bit for bit; rows no present atom of a real residue owns are untouched
    ca = torch.tensor(sorted(ca_rows))
    assert torch.equal(new[ca], xyz[ca])
    assert float(res["max_restraint_dev"].max()) < 1.5          # measured: at most 1.32 A (ragged, member 3)


def test_clash_free_members_padded_rows_and_determinism(states):
    bm, plan, fs, out, planted, _ = _case(states, "ragged", "fp32")
    # members 1 and 3 on a clash-free lattice (slot t of residue i at (10 i, 0, 2 t)), members 0 and 2 decoded with planted clashes
    xyz = planted.cpu().clone()
    for b in (1, 3):
        f = int(fs.frame_of[b])
        for i in range(int(fs.lengths[f])):
            for t in range(14):
                if int(fs.slot_atom[f, i * 14 + t]) >= 0:
                    xyz[_row(fs, b, i, t)] = torch.tensor([10.0 * i, 0.0, 2.0 * t])
    xyz = xyz.cuda()
    thr = THR
    counts, _ = O.repulsion_counts(xyz.cpu(), *_args(fs), O.cutoff(thr))
    clean = [b for b in range(fs.NB) if int(counts[b].sum()) == 0]
    assert clean == [1, 3]
    sentinel = torch.full((xyz.shape[0] + 5, 3), 7.0, device="cuda")
    sentinel[:xyz.shape[0]] = xyz
    a, _, _ = plan.relax(sentinel, thr, sampler.RELAX_ITERATIONS)
    b_, _, _ = plan.relax(sentinel, thr, sampler.RELAX_ITERATIONS)
    assert torch.equal(a, b_), "two calls differ"
    assert torch.equal(a[xyz.shape[0]:], sentinel[xyz.shape[0]:]), "rows past the atoms were written"
    for b in clean:
        o, n = int(fs.out_off[b]), int(fs.num_atoms[int(fs.frame_of[b])])
        assert torch.equal(a[o:o + n], xyz[o:o + n]), b
    assert not torch.equal(a[:int(fs.num_atoms[0])], xyz[:int(fs.num_atoms[0])])
    # a member relaxed alone, in a plan of its own length, equals the same member relaxed in the batch
    prot = synthetic.make_protein(70, 1, seed=2302)
    alone = sampler.frames_from_batch(synthetic.collate(prot), prot.info, 1)
    p1 = bm.upload(alone)
    o, n = int(fs.out_off[1]), int(fs.num_atoms[1])
    assert int(alone.total_atoms) == n and int(fs.frame_of[1]) == 1
    single, _, _ = p1.relax(planted[o:o + n].contiguous(), 1.2, 20)
    batch, _, _ = plan.relax(planted, 1.2, 20)
    assert not torch.equal(single, planted[o:o + n])
    assert torch.equal(single, batch[o:o + n])


def test_edge_pairs_at_the_repulsion_distance(states):
    bm, plan, fs, out, _, _ = _case(states, "ragged", "fp32")
    thr = 0.5
    c = O.cutoff(thr)
    for b, side in ((0, True), (1, False), (2, True), (3, False)):
        xyz = out["xyz"].cpu().clone()
        f = int(fs.frame_of[b])
        n = int(fs.lengths[f])
        i, j = 5, n - 5
        target = xyz[_row(fs, b, j, O.SLOT_CA)]
        inside, outside = _edge_point(target, c)
        beyond = outside.clone()
        beyond[0] = float(np.nextafter(np.float32(beyond[0]), np.float32(np.inf)))
        for point, hit in ((inside, True), (outside, False), (beyond, False)):
            x = xyz.clone()
            x[_last(fs, b, i)] = point
            x = x.cuda()
            d = float(O.pair_dist32(x.cpu(), torch.tensor([[_last(fs, b, i), _row(fs, b, j, O.SLOT_CA)]]))[0])
            assert (d < c) == hit
            plan.relax(x, thr, 1)
            nrep = plan.buffer("relax_nrep").cpu()
            want, _ = O.repulsion_counts(x.cpu(), *_args(fs), c)
            assert torch.equal(nrep[b], torch.where(torch.arange(14) == O.SLOT_CA, 0, want[b])), (point, hit)


# ------------------------------------------------------------------------------------------------ trajectories
_TRAJ = {}


def _traj_bm(states):
    if "bm" not in _TRAJ:
        _TRAJ["bm"] = sampler.Backmapper(*states, "N6", num_sampling_steps="ddim10", precision="fp32", sampler="ddim")
    return _TRAJ["bm"]


def test_backmap_coords_relax_equals_relax_per_pass(states):
    bm = _traj_bm(states)
    prot = synthetic.trajectory(40, 4, seed=77)
    E, opt = 2, {"iterations": 30, "threshold": 1.2}
    plain = bm.backmap_coords(prot.ca_full, prot.restype_full, prot.info, num_ensemble=E, chunks=2, seed=11)
    relaxed = bm.backmap_coords(prot.ca_full, prot.restype_full, prot.info, num_ensemble=E, chunks=2, seed=11, relax=opt)
    for f in range(prot.ca_full.shape[0]):
        fs = sampler.frames_from_coords(prot.ca_full[f:f + 1], prot.restype_full, prot.info, E)
        plan = bm.upload(fs)
        bm.update_coords(plan, fs, prot.ca_full[f:f + 1].cuda())
        dummy = {k: None for k in ("latent", "idx", "zq", "ic_recon")}
        res = bm.relax(plan, fs, dict(dummy, xyz=plain[f].reshape(-1, 3).cuda().contiguous()), **opt)
        assert torch.equal(res["xyz"].cpu().view_as(relaxed[f]), relaxed[f]), f
    assert not torch.equal(plain, relaxed)


def test_sharded_relax_is_independent_of_the_world_size(states):
    bm = _traj_bm(states)
    job = [(p.ca_full, p.restype_full, p.info) for p in (synthetic.trajectory(40, 3, seed=5), synthetic.trajectory(30, 4, seed=6))]
    opt = {"iterations": 20}
    outs = []
    for world in (1, 2, 3):
        merged = None
        for r in range(world):
            o = sampler.ShardedBackmapper(bm, rank=r, world=world).backmap_coords(job, num_ensemble=2, chunks=2, seed=3, relax=opt)
            if merged is None:
                merged = [torch.full_like(t, float("nan")) for t in o]
            for m, t in zip(merged, o):
                mine = ~torch.isnan(t).flatten(1).all(1)
                m[mine] = t[mine]
        outs.append(merged)
    for w in (1, 2):
        for a, b in zip(outs[0], outs[w]):
            assert torch.equal(a, b), w
