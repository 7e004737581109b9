"""GPU tests of clash-driven repair (run on the B200 box: pytest -m gpu): the per-residue clash counts and keep masks of
cb2_plan_residue_clashes against the brute-force CPU oracle (tests/clash_oracle.py), bit for bit, on decoded samples of both
tiers, on planted clashes far apart in sequence and space, and at the threshold's edge; the counts against cb2_pair_losses; and
the properties of Backmapper.repair under DDPM and DDIM."""
import numpy as np
import pytest
import torch

from codlad_b200 import metrics, sampler, synthetic, weights
from codlad_b200.sampler import clash_pair_totals
from oracle.restate import _pd
from tests import clash_oracle as O
from tests import parity_utils as P
from tests.test_gpu_ddim import _inputs

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

THRESHOLDS = (1.2, 2.5, 3.5)
GROWS = (0, 1, 8)


@pytest.fixture(scope="module")
def states():
    return weights.init_denoiser_state(0), weights.init_vae_decode_state(0)


def _frameset(case):
    """The golden / ragged inputs of the DDIM and inpainting tests, with the topology of the proteins they were built from."""
    inp = _inputs(case)
    if case == "golden":
        L, prot_seed = (int(v) for v in P.golden("sampler_L64_100")["meta"][:2])
        prots = [synthetic.make_protein(L, 1, seed=prot_seed)]
        batch = synthetic.collate(prots[0])
    else:
        prots = [synthetic.make_protein(n, 1, seed=2301 + b) for b, n in enumerate((80, 70))]
        batch = synthetic.collate_many(prots)
    fs = sampler.frames_from_batch(batch, [p.info for p in prots], frame_of=inp["frame_of"])
    assert torch.equal(fs.X, inp["X"])
    return fs, inp


def _decoded(states, case, precision):
    fs, inp = _frameset(case)
    bm = sampler.Backmapper(*states, "N6", num_sampling_steps=10, precision=precision)
    plan = bm.upload(fs)
    out = bm.sample(plan, fs, inp["z0"], inp["noises"][:10].contiguous())
    return bm, plan, fs, out


def _check_vs_oracle(bm, plan, fs, xyz, thresholds=THRESHOLDS):
    nbr = plan.buffer("nbr_idx").cpu()
    total = 0
    for thr in thresholds:
        want = O.residue_clashes(xyz.cpu(), fs.slot_atom, fs.out_off, fs.lengths, fs.frame_of, fs.L, thr)
        total += int(want.sum())
        for grow in GROWS:
            counts, keep = bm.residue_clashes(plan, fs, xyz, thr, grow)
            assert counts.dtype == torch.int32 and keep.dtype == torch.bool and counts.shape == keep.shape == (fs.NB, fs.L)
            assert torch.equal(counts.cpu(), want), (thr, grow)
            assert torch.equal(keep.cpu(), O.keep_mask(want, nbr, fs.lengths, fs.frame_of, grow)), (thr, grow)
    return total


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("case", ["golden", "ragged"])
def test_counts_and_keep_vs_oracle(states, case, precision):
    bm, plan, fs, out = _decoded(states, case, precision)
    assert _check_vs_oracle(bm, plan, fs, out["xyz"]) > 0, "no clash at any threshold: the case tests nothing"


def _edge_point(a, thr):
    """An fp32 point on the x line through atom a whose distance to a, as _pd forms it, is the largest one below thr, and the next
    fp32 point outward (distance >= thr)."""
    x = np.float32(float(a[0]) + thr)
    point = lambda v: torch.tensor([float(v), float(a[1]), float(a[2])])
    d = lambda v: float(_pd(torch.stack((a, point(v))), torch.tensor([[0, 1]]))[0])
    while d(x) >= thr:
        x = np.nextafter(x, np.float32(-np.inf))
    return point(x), point(np.nextafter(x, np.float32(np.inf)))


def test_planted_far_clashes_and_threshold_edges(states):
    """Clashes planted between residues far apart in sequence and outside each other's k-NN rows, by moving a side-chain atom
    more than 10 Angstrom away from its C-alpha (the bounding spheres must grow with it), and pairs one fp32 step on either side of
    the threshold."""
    bm, plan, fs, out = _decoded(states, "ragged", "fp32")
    xyz = out["xyz"].cpu().clone()
    nbr = plan.buffer("nbr_idx").cpu()
    ca = lambda b, i: int(fs.out_off[b]) + int(fs.slot_atom[int(fs.frame_of[b]), i * 14 + 3])
    last = lambda b, i: int(fs.out_off[b]) + int(fs.slot_atom[int(fs.frame_of[b]), i * 14:(i + 1) * 14].max())
    planted = []
    for b in range(fs.NB):
        f, n = int(fs.frame_of[b]), int(fs.lengths[int(fs.frame_of[b])])
        side = [r for r in range(n) if int(fs.slot_atom[f, r * 14 + 4]) >= 0]        # residues with a side chain
        for i, shift in ((side[b], 0.4), (side[-1 - b], None)):
            d = (xyz[[ca(b, j) for j in range(n)]] - xyz[ca(b, i)]).norm(dim=1)
            j = int(d.argmax())
            assert j not in nbr[f, i].tolist() and abs(i - j) > 8
            if shift is not None:
                xyz[last(b, i)] = xyz[ca(b, j)] + torch.tensor([shift, 0.0, 0.0])
            else:                                 # threshold edge: inside on even members, outside on odd ones
                inside, outside = _edge_point(xyz[ca(b, j)], 1.2)
                xyz[last(b, i)] = inside if b % 2 == 0 else outside
            assert float((xyz[last(b, i)] - xyz[ca(b, i)]).norm()) > 10.0
            planted.append((b, i, j, shift is not None or b % 2 == 0))
    xyz = xyz.cuda()
    _check_vs_oracle(bm, plan, fs, xyz, (1.2,))
    counts, keep = bm.residue_clashes(plan, fs, xyz, 1.2, 0)
    for b, i, j, hit in planted:
        if hit:
            assert counts[b, i] > 0 and counts[b, j] > 0 and not keep[b, i] and not keep[b, j]


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_counts_equal_pair_losses(states, precision):
    """For the 64-residue member, half the summed counts equal cb2_pair_losses' count over all inter-residue, non-peptide pairs."""
    bm, plan, fs, out = _decoded(states, "golden", precision)
    pairs = O.unordered_pairs(fs.slot_atom, fs.out_off, fs.lengths, fs.frame_of, 0, fs.L).cuda()
    for thr in THRESHOLDS:
        counts, _ = bm.residue_clashes(plan, fs, out["xyz"], thr)
        assert int(counts.sum()) % 2 == 0
        assert int(counts.sum()) // 2 == int(metrics.pair_losses(out["xyz"], pairs, thr_count=thr)[0])


def test_residue_clashes_rejects_bad_arguments(states):
    bm, plan, fs, out = _decoded(states, "golden", "fp32")
    xyz = out["xyz"]
    for bad in (xyz[:-1], xyz.double(), xyz.cpu(), xyz[:, :2]):
        with pytest.raises(ValueError):
            bm.residue_clashes(plan, fs, bad)
    for thr, grow in ((0.0, 0), (float("nan"), 0), (1.2, -1), (1.2, plan.K)):
        with pytest.raises(ValueError):
            bm.residue_clashes(plan, fs, xyz, thr, grow)
    with pytest.raises(ValueError):
        bm.repair(plan, fs, out, max_rounds=-1)
    with pytest.raises(ValueError):
        bm.repair(plan, fs, {"xyz": xyz})


# ------------------------------------------------------------------------------------------------ the repair loop
NB_REPAIR, L_REPAIR = 6, 120


def _repair_case(states, kind):
    prot = synthetic.make_protein(L_REPAIR, 1, seed=1011)
    fs = sampler.frames_from_batch(synthetic.collate(prot), prot.info, NB_REPAIR)
    bm = sampler.Backmapper(*states, "N6", num_sampling_steps=25, precision="f16", sampler=kind)
    z, sn = synthetic.latent_noise((NB_REPAIR, L_REPAIR, 3), 3011), synthetic.latent_noise((25, NB_REPAIR, L_REPAIR, 3), 3012)
    return bm, fs, z, sn


def _mixed_threshold(fs, xyz):
    """A threshold at which about half of the members clash: halfway between two members' closest inter-residue pairs (the
    synthetic weights may give more or fewer clashes at 1.2 A than real ones; this makes the loop run and leaves members alone)."""
    m = []
    for b in range(fs.NB):
        pairs = O.unordered_pairs(fs.slot_atom, fs.out_off, fs.lengths, fs.frame_of, b, fs.L)
        m.append(float(_pd(xyz.cpu(), pairs).min()))
    m = sorted(m)
    k = len(m) // 2
    assert m[k - 1] < m[k]
    return (m[k - 1] + m[k]) / 2


def _member_rows(fs, b):
    o = int(fs.out_off[b])
    return slice(o, o + int(fs.num_atoms[int(fs.frame_of[b])]))


@pytest.mark.parametrize("kind", ["ddpm", "ddim"])
def test_repair_loop(states, kind):
    bm, fs, z, sn = _repair_case(states, kind)
    plan = bm.upload(fs)
    first = {k: v.clone() for k, v in bm.sample(plan, fs, z, sn).items()}
    thr = _mixed_threshold(fs, first["xyz"])
    counts0, keep0 = bm.residue_clashes(plan, fs, first["xyz"], thr)
    pairs0 = clash_pair_totals(counts0)
    clean = [b for b in range(fs.NB) if int(pairs0[b]) == 0]
    assert 0 < len(clean) < fs.NB
    print(f"repair {kind}: threshold {thr:.3f} A, input clash pairs per member {pairs0.tolist()}")

    # max_rounds = 0: the input, bit for bit
    same = bm.repair(plan, fs, {k: v.clone() for k, v in first.items()}, max_rounds=0, threshold=thr)
    for k in first:
        assert torch.equal(same[k], first[k]), k
    assert torch.equal(same["clashes"], counts0) and same["clash_pairs"].tolist() == [pairs0.tolist()]

    # one round: every residue kept in it keeps its latent and VQ index
    gen = torch.Generator(device="cuda").manual_seed(5)
    one = bm.repair(plan, fs, {k: v.clone() for k, v in first.items()}, max_rounds=1, threshold=thr, generator=gen)
    assert one["clash_pairs"].shape == (2, fs.NB)
    assert torch.equal(one["latent"][keep0], first["latent"][keep0])
    assert torch.equal(one["idx"][keep0], first["idx"][keep0])

    # three rounds
    gen = torch.Generator(device="cuda").manual_seed(7)
    res = bm.repair(plan, fs, {k: v.clone() for k, v in first.items()}, max_rounds=3, threshold=thr, generator=gen)
    cp = res["clash_pairs"].cpu()
    print(f"repair {kind}: clash pairs per round {cp.tolist()}")
    assert cp.dtype == torch.int64 and 2 <= cp.shape[0] <= 4 and cp.shape[1] == fs.NB
    assert torch.equal(cp[0], pairs0.cpu())
    assert bool((cp[1:] <= cp[:-1]).all()), "a member's clash count went up"
    want, _ = bm.residue_clashes(plan, fs, res["xyz"], thr)
    assert torch.equal(res["clashes"], want)
    assert torch.equal(clash_pair_totals(res["clashes"]).cpu(), cp[-1])
    for b in clean:
        assert torch.equal(res["latent"][b], first["latent"][b]), b
        assert torch.equal(res["idx"][b], first["idx"][b]), b
        assert torch.equal(res["xyz"][_member_rows(fs, b)], first["xyz"][_member_rows(fs, b)]), b

    # the plan is left for a plain pass: sample() equals a fresh Backmapper's
    again = bm.sample(plan, fs, z, sn)
    bm2 = sampler.Backmapper(*states, "N6", num_sampling_steps=25, precision="f16", sampler=kind)
    fresh = bm2.sample(bm2.upload(fs), fs, z, sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(again[k], fresh[k]), k
        assert torch.equal(again[k], first[k]), k
