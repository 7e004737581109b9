"""CPU tests of trajectory backmapping from a coordinate array: the topology FrameSet of Backmapper.backmap_coords against
frames_from_batch, the host radius graph (the form the device graph is compared with on the GPU) against a float64 restatement of
the rule, and the argument checks of backmap_coords, update_coords and Plan.set_coords that run before any device call."""
import numpy as np
import pytest
import torch

from codlad_b200 import batching, synthetic
from codlad_b200.engine import Plan
from codlad_b200.sampler import Backmapper, FrameSet, frames_from_batch, frames_from_coords


def _coords_and_batch(prot, frames):
    return prot.ca_full[frames].contiguous(), synthetic.collate(prot, frames)


@pytest.mark.parametrize("num_ensemble", [1, 3])
@pytest.mark.parametrize("frames", [[0], [2, 0, 4]])
def test_frames_from_coords_equals_frames_from_batch(frames, num_ensemble):
    prot = synthetic.trajectory(37, 5, seed=11)
    ca, batch = _coords_and_batch(prot, frames)
    got = frames_from_coords(ca, prot.restype_full, prot.info, num_ensemble)
    want = frames_from_batch(batch, prot.info, num_ensemble)
    for name in ("X", "ca_full", "cg_z", "lengths", "orders", "slot_atom", "num_atoms", "frame_of", "out_off"):
        a, b = getattr(got, name), getattr(want, name)
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b), name
    assert got.total_atoms == want.total_atoms
    assert got.csr_row.shape == want.csr_row.shape and not bool(got.csr_row.any()) and got.csr_col.numel() == 0


def _restated_csr(X: np.ndarray, cutoff: float):
    """The radius rule in float64 (no rounding to fp32 on the way), one frame: (row_ptr, col, |d - cutoff| of every pair)."""
    d = np.sqrt(((X[None, :, :] - X[:, None, :]) ** 2).sum(-1))
    keep = d <= cutoff
    np.fill_diagonal(keep, False)
    counts = keep.sum(1)
    row_ptr = np.concatenate([[0], np.cumsum(counts)])
    col = np.concatenate([np.nonzero(r)[0] for r in keep]) if keep.any() else np.zeros(0, dtype=np.int64)
    return row_ptr, col, np.abs(d - cutoff)


@pytest.mark.parametrize("case", ["walk40", "walk300", "compact200", "one"])
def test_host_radius_graph_follows_the_rule(case):
    """batching.batch_csr(synthetic.radius_graph(...)) against the float64 rule: equal, apart from rows holding a pair within
    1e-5 A of the cutoff (where fp32 rounding may decide either way)."""
    L, compact = {"walk40": (40, 0.0), "walk300": (300, 0.0), "compact200": (200, 0.6), "one": (1, 0.0)}[case]
    prot = synthetic.make_protein(L, 2, seed=77, compact=compact)
    batch = synthetic.collate(prot)
    row_ptr, col = batching.batch_csr(batch["CG_nbr_list"], batch["num_CGs"], L)
    ambiguous = 0
    for f in range(2):
        X = prot.ca_full[f, 1:-1].double().numpy()
        rp, cl, gap = _restated_csr(X, synthetic.CG_CUTOFF)
        base = int(row_ptr[f * L])
        for i in range(L):
            got = col[int(row_ptr[f * L + i]):int(row_ptr[f * L + i + 1])].numpy()
            want = cl[rp[i]:rp[i + 1]]
            near = np.delete(gap[i], i) < 1e-5
            if near.any():
                ambiguous += 1
                continue
            assert np.array_equal(got, want), (f, i)
        assert base == (0 if f == 0 else int(row_ptr[L]))
    if case == "compact200":
        assert int(row_ptr[-1]) / (2 * L) > 50            # the compact walk is dense
    print(f"{case}: {int(row_ptr[-1])} edges, {ambiguous} rows with a pair within 1e-5 A of the cutoff")


# ---- argument checks (no device is touched) -------------------------------------------------------------------------------------
def _bm(T=10):
    bm = object.__new__(Backmapper)          # the checks below run before any use of the engines
    bm.T = T
    return bm


def _traj(n=4, L=12):
    prot = synthetic.trajectory(L, n, seed=3)
    return prot.ca_full.contiguous(), prot.restype_full, prot.info


@pytest.mark.parametrize("kw", [dict(num_ensemble=0), dict(num_ensemble=True), dict(num_ensemble=1.0), dict(steps=0), dict(steps=11),
                                dict(steps=1.5), dict(chunks=0), dict(chunks=5), dict(chunks=2.0), dict(chunks=True)])
def test_backmap_coords_rejects_arguments(kw):
    ca, rt, info = _traj()
    with pytest.raises(ValueError):
        _bm().backmap_coords(ca, rt, info, **kw)


def test_backmap_coords_rejects_coordinates_and_restype():
    ca, rt, info = _traj()
    bad = [(ca.double(), rt), (ca[..., :2], rt), (ca[0], rt), (ca[:0], rt), (ca[:, :2], rt[:2]), (ca.to("meta"), rt),
           (ca.numpy(), rt), (ca, rt[:-1]), (ca, rt.float()), (ca, rt.bool()), (ca, rt[None])]
    for c, r in bad:
        with pytest.raises(ValueError):
            _bm().backmap_coords(c, r, info)


def _fake_plan(fs: FrameSet, device="cuda"):
    return type("P", (), {"device": torch.device(device, 0), "F": fs.F, "NB": fs.NB, "L": fs.L})()


def test_update_coords_rejects():
    ca, rt, info = _traj()
    fs = frames_from_coords(ca[:2], rt, info, 3)
    plan = _fake_plan(fs)
    for bad in (ca[:2], ca[:2].double(), ca[:3], ca[:2, :-1], ca[:2, :, :2], ca[:2].numpy()):
        with pytest.raises(ValueError):
            _bm().update_coords(plan, fs, bad)                # a host tensor, wrong dtype or shape
    other = frames_from_coords(ca[:3], rt, info, 1)
    with pytest.raises(ValueError, match="shape|frame set"):
        _bm().update_coords(_fake_plan(other), fs, ca[:2].to("meta"))


def test_plan_set_coords_rejects():
    plan = object.__new__(Plan)
    plan.F, plan.NB, plan.L, plan.device = 2, 2, 12, torch.device("cuda", 0)
    ca = torch.zeros(2, 14, 3)
    for bad in (ca, ca.double(), ca[:1], ca[:, :13], ca.numpy(), None):
        with pytest.raises(ValueError):
            plan.set_coords(None, bad)
