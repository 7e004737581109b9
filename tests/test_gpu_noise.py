"""GPU tests of the keyed sampling noise (run on the B200 box: pytest -m gpu): engine.keyed_normal against the float64 restatement
(tests/noise_oracle.py), its invariance to the batch (bit for bit), its statistics, the seeded Backmapper paths against the
explicit-noise paths (bit for bit), a member alone against the same member in a ragged batch and the sharded driver against one
GPU (within the tier bars, with bit identity recorded), the refusals and the launch count."""
import ctypes as C

import numpy as np
import pytest
import torch

from codlad_b200 import synthetic, weights
from tests import noise_oracle as O
from tests import parity_utils as P

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

BARS = {"fp32": 1.5e-6, "f16": 1.5e-3}
SEED = 0x5EED_0000_C0DE_0001
VARIANTS = {"ddpm10": ("ddpm", "10", 0.0), "ddim50_eta0": ("ddim", "ddim50", 0.0), "ddim50_eta1": ("ddim", "ddim50", 1.0)}


@pytest.fixture(scope="module")
def eng():
    from codlad_b200 import engine
    return engine


_BMS = {}


def _bm(precision="f16", variant="ddpm10"):
    from codlad_b200 import sampler as S
    key = (precision, variant)
    if key not in _BMS:
        sampler, steps, eta = VARIANTS[variant]
        _BMS[key] = S.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=steps,
                                 precision=precision, sampler=sampler, eta=eta)
    return _BMS[key]


def _proteins(lengths):
    return [synthetic.make_protein(n, 1, seed=500 + 7 * i + n) for i, n in enumerate(lengths)]


def _fs(proteins, num_ensemble=1, frame_of=None):
    from codlad_b200 import sampler as S
    return S.frames_from_batch(synthetic.collate_many(proteins, 0), [p.info for p in proteins], num_ensemble, frame_of=frame_of)


def _keys(vals):
    return torch.tensor(vals, dtype=torch.int64, device="cuda")


def _clone(out):
    return {k: v.clone() for k, v in out.items() if torch.is_tensor(v)}


# ---- 1. the fill ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["L300x3", "L1x1", "L7x5_high_slices", "big_keys"])
def test_fill_against_the_restatement(eng, case):
    keys, L, draw, first, n, seed = {
        "L300x3": ([0, 1, 65536 + 2], 300, 0, 0, 101, SEED),
        "L1x1": ([123], 1, 7, 0, 3, 0),
        "L7x5_high_slices": ([5, 4, 3, 2, 1], 7, 2 ** 32 - 1, 2000, 48, 2 ** 64 - 1),
        "big_keys": ([2 ** 63 - 1, -1, -(2 ** 63), (2 ** 47 - 1) * 65536 + 65535], 2048, 1, 100, 2, 12345),
    }[case]
    got = eng.keyed_normal(seed, _keys(keys), L, draw, first, n).cpu().double().numpy()
    want = O.keyed_normal(seed, keys, L, draw, first, n)
    assert got.shape == want.shape == (n, len(keys), L, 3)
    err = np.abs(got - want)
    worst = np.unravel_index(int(err.argmax()), err.shape)
    print(f"keyed_normal {case}: {got.size} values, worst |gpu - float64| {err.max():.3e} at {worst} (value {want[worst]:+.6f}), "
          f"max |value| {np.abs(want).max():.3f}")
    assert np.isfinite(got).all()
    assert err.max() < 1e-5


def test_fill_at_the_largest_row_index(eng):
    """Row i = 2^21 - 1 (the largest the counter's row field holds) of a one-slice fill, against the restatement."""
    L = 2 ** 21 - 1
    got = eng.keyed_normal(SEED, _keys([9]), L, 0, 2047, 1)[0, 0, -4:].cpu().double().numpy()
    want = O.keyed_normal(SEED, [9], L, 0, 2047, 1)[0, 0, -4:]
    assert np.abs(got - want).max() < 1e-5


# ---- 2. invariance ---------------------------------------------------------------------------------------------------------------
def test_member_slices_do_not_depend_on_the_batch(eng):
    keys = [f * 65536 + e for e in range(2) for f in range(5)]                                   # 10 members
    full = eng.keyed_normal(SEED, _keys(keys), 300, 3, 0, 101)
    for b in (0, 4, 9):
        alone = eng.keyed_normal(SEED, _keys([keys[b]]), 300, 3, 0, 101)
        assert torch.equal(alone[:, 0], full[:, b])
    perm = torch.randperm(10, generator=torch.Generator().manual_seed(1))
    permuted = eng.keyed_normal(SEED, _keys([keys[p] for p in perm.tolist()]), 300, 3, 0, 101)
    assert torch.equal(permuted, full[:, perm.cuda()])
    padded = eng.keyed_normal(SEED, _keys(keys), 320, 3, 0, 101)
    assert torch.equal(padded[:, :, :300], full)
    assert not torch.equal(eng.keyed_normal(SEED, _keys(keys), 300, 4, 0, 101), full)


def test_partial_fills_equal_full_fills(eng):
    keys = _keys([7, 8, 65536 * 3])
    full = eng.keyed_normal(SEED, keys, 50, 1, 0, 101)
    for first, n in ((0, 1), (1, 100), (1, 50), (51, 50), (37, 1), (100, 1)):
        assert torch.equal(eng.keyed_normal(SEED, keys, 50, 1, first, n), full[first:first + n]), (first, n)
    out = torch.full((101, 3, 50, 3), float("nan"), device="cuda")
    eng.keyed_normal(SEED, keys, 50, 1, 0, 1, out=out[:1])
    eng.keyed_normal(SEED, keys, 50, 1, 1, 100, out=out[1:])
    assert torch.equal(out, full)


# ---- 3. statistics ----------------------------------------------------------------------------------------------------------------
def test_statistics(eng):
    from scipy import stats
    S, NB, L = 64, 1024, 256                        # 2^24 rows, 3 * 2^24 values
    keys = _keys(list(range(NB)))
    a = eng.keyed_normal(SEED, keys, L, 0, 0, S).double()
    n = a.numel()
    mean, var = float(a.mean()), float(a.var())
    z_mean, z_var = mean * n ** 0.5, (var - 1.0) / (2.0 / n) ** 0.5
    flat = a.flatten()[: 1 << 24].cpu().numpy()
    ks = stats.kstest(flat, "norm")

    def corr(x, y):
        x, y = x.flatten() - x.mean(), y.flatten() - y.mean()
        return float((x * y).sum() / (x.norm() * y.norm()))

    ch = {f"ch{i}-ch{j}": corr(a[..., i], a[..., j]) for i, j in ((0, 1), (0, 2), (1, 2))}
    adj_key = corr(a[:, :-1], a[:, 1:])
    adj_slice = corr(a[:-1], a[1:])
    del a
    b = eng.keyed_normal(SEED, keys, L, 1, 0, S).double()
    adj_draw = corr(eng.keyed_normal(SEED, keys, L, 0, 0, S).double(), b)
    print(f"statistics over {n} values: mean {mean:+.3e} ({z_mean:+.2f} sigma), variance {var:.6f} ({z_var:+.2f} sigma), "
          f"KS p = {ks.pvalue:.3g} over {flat.size}, correlations {', '.join(f'{k} {v:+.2e}' for k, v in ch.items())}, "
          f"adjacent keys {adj_key:+.2e}, adjacent slices {adj_slice:+.2e}, adjacent draws {adj_draw:+.2e}")
    assert abs(z_mean) < 5 and abs(z_var) < 5
    assert ks.pvalue > 1e-4
    for v in list(ch.values()) + [adj_key, adj_slice, adj_draw]:
        assert abs(v) < 1e-3


# ---- 4. seeded path = explicit-noise path ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("mode", ["sample", "refine"])
def test_seeded_equals_explicit_noise(eng, mode, variant, precision):
    from codlad_b200 import sampler as S
    bm = _bm(precision, variant)
    fs = _fs(_proteins((80, 70, 40)), frame_of=[0, 1, 2, 1])
    plan = bm.upload(fs)
    T = bm.T
    keys = S.member_keys(fs).cuda()
    fill = eng.keyed_normal(SEED, keys, fs.L, 2, 0, 1 + T)
    noisy = variant != "ddim50_eta0"
    if mode == "sample":
        bm.sample(plan, fs, seed=SEED + 2)                             # capture the graph
        l0 = plan.launches
        got = _clone(bm.sample(plan, fs, seed=SEED, draw=2))
        l1 = plan.launches
        want = _clone(bm.sample(plan, fs, z=fill[0], step_noise=fill[1:] if noisy else None))
        assert plan.launches - l1 == l1 - l0
    else:
        base = _clone(bm.sample(plan, fs, seed=SEED + 1))
        got = _clone(bm.refine(plan, fs, base["latent"], T // 2, seed=SEED, keys=keys.cpu(), draw=2))
        want = _clone(bm.refine(plan, fs, base["latent"], T // 2, z=fill[0], step_noise=fill[1:] if noisy else None))
    for k in ("latent", "idx", "xyz"):
        assert torch.equal(got[k], want[k]), k
    again = _clone(bm.sample(plan, fs, seed=SEED, draw=2)) if mode == "sample" else \
        _clone(bm.refine(plan, fs, base["latent"], T // 2, seed=SEED, keys=keys, draw=2))
    assert torch.equal(again["latent"], got["latent"]) and torch.equal(again["xyz"], got["xyz"])


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_seeded_repeat_runs_and_launch_count(precision):
    bm = _bm(precision, "ddpm10")
    fs = _fs(_proteins((60, 45)), num_ensemble=3)
    plan = bm.upload(fs)
    bm.sample(plan, fs)                                                 # capture the graph
    l0 = plan.launches
    bm.sample(plan, fs, generator=torch.Generator(device="cuda").manual_seed(0))
    l1 = plan.launches
    a = _clone(bm.sample(plan, fs, seed=SEED))
    l2 = plan.launches
    b = _clone(bm.sample(plan, fs, seed=SEED))
    assert l1 - l0 == l2 - l1 == plan.launches - l2
    for k in a:
        assert torch.equal(a[k], b[k]), k
    c = _clone(bm.sample(plan, fs, seed=SEED + 1))
    assert not torch.equal(a["latent"], c["latent"])


# ---- 5. a member alone against the same member in a batch ----------------------------------------------------------------------
# The model itself depends on the padded length L, as the reference does: the local frames of the orientation features exist for
# residues 1 .. L-3 of the padded length (protein_mpnn_utils.py:397-426, oracle.restate.residue_frames), so the last residues of a
# frame padded further see other features.  A member alone is therefore compared at its batch's padded length: its frame is planned
# together with the batch's longest frame, which no member uses.
@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("case", ["ragged", "K40"])
def test_member_alone_against_the_batch(precision, case):
    from codlad_b200 import sampler as S
    bm = _bm(precision, "ddpm10")
    prots = _proteins((80, 70, 40) if case == "ragged" else (40, 40, 40))
    frame_of = [0, 1, 2, 1]
    fs = _fs(prots, frame_of=frame_of)
    keys = S.member_keys(fs)
    plan = bm.upload(fs)
    batch = _clone(bm.sample(plan, fs, seed=SEED))
    worst, identical = 0.0, []
    for b, f in enumerate(frame_of):
        one = _fs([prots[f]] if f == 0 else [prots[f], prots[0]], frame_of=[0])
        n = prots[f].L
        alone = _clone(bm.sample(bm.upload(one), one, seed=SEED, keys=keys[b:b + 1]))
        err = P.rel_err(alone["latent"][0, :n].cpu(), batch["latent"][b, :n].cpu())
        same = torch.equal(alone["latent"][0, :n], batch["latent"][b, :n])
        flips = int((alone["idx"][0, :n] != batch["idx"][b, :n]).sum())
        print(f"{precision} {case} member {b} (frame L={n}, plan L={fs.L}, K={plan.K}): latent rel err {err:.3e}, "
              f"bit-identical {same}, VQ flips {flips}/{n}")
        worst = max(worst, err)
        identical.append(same)
        assert err < BARS[precision], (b, err)
    print(f"{precision} {case}: worst latent rel err {worst:.3e}; bit-identical members {sum(identical)}/{len(identical)}")


# ---- 6. the sharded driver ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_sharded_against_one_gpu(precision):
    """Lengths 60 / 60 / 50 x 2 members: world 1 plans all three frames together, world 2 plans frames {0, 2} and {1}; every group
    is padded to 60, so each unit sees the model at the same L and only its batch changes."""
    from codlad_b200 import sampler as S
    bm = _bm(precision, "ddpm10")
    prots = _proteins((60, 60, 50))
    batches = [synthetic.collate(p) for p in prots]
    infos = [p.info for p in prots]
    lengths = [p.L for p in prots]
    one = S.ShardedBackmapper(bm, rank=0, world=1)
    ref = one.backmap_local(batches, infos, one.plan(lengths, 2)[0], lengths, seed=SEED)
    got = {}
    for r in range(2):
        sb = S.ShardedBackmapper(bm, rank=r, world=2)
        parts = sb.plan(lengths, 2)
        print(f"{precision} rank {r}/2: units {parts[r]}, groups {[g[0] for g in sb.local_groups(parts[r], lengths)]}; "
              f"world 1 groups {[g[0] for g in one.local_groups(one.plan(lengths, 2)[0], lengths)]}")
        got.update(sb.backmap_local(batches, infos, parts[r], lengths, seed=SEED))
    assert sorted(got) == sorted(ref) == [(f, e) for f in range(3) for e in range(2)]
    same, worst = 0, 0.0
    for u in ref:
        err = P.rel_err(got[u], ref[u])
        same += int(torch.equal(got[u], ref[u]))
        worst = max(worst, err)
        assert err < BARS[precision], (u, err)
    print(f"{precision}: sharded (world 2) against world 1, worst coordinate rel err {worst:.3e}, bit-identical units "
          f"{same}/{len(ref)}")
    # and the units' noise is the one a single-GPU run of the whole job with member_keys draws
    fs = _fs(prots, num_ensemble=2)
    assert S.member_keys(fs).tolist() == [f * 65536 + e for e in range(2) for f in range(3)]


def test_sharded_backmap_world_one_passes_the_seed():
    from codlad_b200 import sampler as S
    bm = _bm("fp32", "ddpm10")
    prots = _proteins((30, 20))
    batches = [synthetic.collate(p) for p in prots]
    infos = [p.info for p in prots]
    sb = S.ShardedBackmapper(bm, rank=0, world=1)
    a = sb.backmap(batches, infos, 2, seed=SEED)
    b = sb.backmap_local(batches, infos, sb.plan([30, 20], 2)[0], [30, 20], seed=SEED)
    assert all(torch.equal(a[u], b[u]) for u in b)


# ---- 7. repair and trajectories -------------------------------------------------------------------------------------------------
def test_seeded_repair_draws_round_by_round(eng):
    """Round r of a seeded repair is resample() with the keyed noise of draw r + 1; two seeded repairs are identical."""
    from codlad_b200 import sampler as S
    bm = _bm("fp32", "ddpm10")
    fs = _fs(_proteins((50, 40)), num_ensemble=2)
    plan = bm.upload(fs)
    out = _clone(bm.sample(plan, fs, seed=SEED))
    r1 = bm.repair(plan, fs, out, max_rounds=2, threshold=3.0, seed=SEED)
    r1 = {k: v.clone() for k, v in r1.items()}
    r2 = bm.repair(plan, fs, out, max_rounds=2, threshold=3.0, seed=SEED)
    assert r1["clash_pairs"].shape[0] > 1, "the threshold flags no clash: the rounds were not exercised"
    for k in ("latent", "xyz", "clash_pairs"):
        assert torch.equal(r1[k], r2[k]), k
    counts, keep = bm.residue_clashes(plan, fs, out["xyz"], 3.0)
    first = _clone(bm.resample(plan, fs, out["latent"], keep, seed=SEED, draw=1))
    keys = S.member_keys(fs).cuda()
    fill = eng.keyed_normal(SEED, keys, fs.L, 1, 0, 1 + bm.T)
    want = _clone(bm.resample(plan, fs, out["latent"], keep, z=fill[0], step_noise=fill[1:]))
    assert torch.equal(first["latent"], want["latent"])


@pytest.mark.parametrize("method", ["trajectory", "coords"])
def test_seeded_trajectory_noise_follows_the_frame(method):
    """backmap_trajectory / backmap_coords with a seed: the first frame of every run is sample() with keys f * 2^16 + e and draw 0,
    whatever `chunks` is; the same call twice gives the same result."""
    from codlad_b200 import sampler as S
    bm = _bm("fp32", "ddpm10")
    traj = synthetic.trajectory(30, 6, seed=3)
    batches = [synthetic.collate(traj, [f]) for f in range(6)]

    def run(chunks):
        if method == "trajectory":
            return bm.backmap_trajectory(batches, traj.info, num_ensemble=2, steps=3, chunks=chunks, seed=SEED)
        return bm.backmap_coords(traj.ca_full, traj.restype_full, traj.info, num_ensemble=2, steps=3, chunks=chunks, seed=SEED)

    three = run(3)                                      # runs start at frames 0, 2, 4
    assert torch.equal(three, run(3))
    one = run(1)
    for f in (0, 2, 4):
        fs = S.frames_from_batch(batches[f], traj.info, 2)
        plan = bm.upload(fs)
        keys = S.member_keys(fs, [f])
        alone = bm.sample(plan, fs, seed=SEED, keys=keys)["xyz"].view(2, -1, 3).cpu()
        assert P.rel_err(three[f], alone) < BARS["fp32"], f
    fs = S.frames_from_batch(batches[0], traj.info, 2)
    assert torch.equal(one[0], bm.sample(bm.upload(fs), fs, seed=SEED)["xyz"].view(2, -1, 3).cpu())


# ---- 8. refusals -----------------------------------------------------------------------------------------------------------------
def test_refusals(eng):
    from codlad_b200 import _native as N
    keys = _keys([1, 2])
    out = torch.empty(2, 2, 5, 3, device="cuda")
    with pytest.raises(ValueError, match="keys"):
        eng.keyed_normal(1, keys.cpu(), 5, 0, 0, 2)
    with pytest.raises(ValueError, match="keys"):
        eng.keyed_normal(1, keys.int(), 5, 0, 0, 2)
    with pytest.raises(ValueError, match="keys"):
        eng.keyed_normal(1, keys[:0], 5, 0, 0, 2)
    with pytest.raises(ValueError, match="out"):
        eng.keyed_normal(1, keys, 5, 0, 0, 3, out=out)
    with pytest.raises(ValueError, match="out"):
        eng.keyed_normal(1, keys, 5, 0, 0, 2, out=out.double())
    with pytest.raises(ValueError, match="out"):
        eng.keyed_normal(1, keys, 5, 0, 0, 2, out=torch.empty(2, 5, 2, 3, device="cuda").transpose(1, 2))
    with pytest.raises(ValueError, match="slices"):
        eng.keyed_normal(1, keys, 5, 0, 2000, 49)
    lib, p, o = N.lib(), N.dptr(keys), N.dptr(out)
    for args, msg in [((1, None, 2, 5, 0, 0, 2, o, None), "null"), ((1, p, 2, 5, 0, 0, 2, None, None), "null"),
                      ((1, p, 0, 5, 0, 0, 2, o, None), "NB"), ((1, p, 2, 0, 0, 0, 2, o, None), "L="),
                      ((1, p, 2, 1 << 21, 0, 0, 2, o, None), "L="), ((1, p, 2, 5, 0, -1, 2, o, None), "slices"),
                      ((1, p, 2, 5, 0, 0, 0, o, None), "slices"), ((1, p, 2, 5, 0, 2047, 2, o, None), "slices")]:
        assert lib.cb2_keyed_normal(*args) != 0, args
        assert msg in lib.cb2_last_error().decode(), (args, lib.cb2_last_error())
    assert lib.cb2_keyed_normal(C.c_uint64(2 ** 64 - 1), p, 2, 5, C.c_uint32(2 ** 32 - 1), 2046, 2, o, None) == 0
    torch.cuda.synchronize()
    bm = _bm("fp32", "ddpm10")
    fs = _fs(_proteins((20,)), num_ensemble=2)
    plan = bm.upload(fs)
    with pytest.raises(ValueError, match="excludes"):
        bm.sample(plan, fs, seed=1, generator=torch.Generator(device="cuda"))
    with pytest.raises(ValueError, match="excludes"):
        bm.sample(plan, fs, seed=1, z=torch.zeros(2, 20, 3, device="cuda"))
    with pytest.raises(ValueError, match="excludes"):
        bm.refine(plan, fs, torch.zeros(2, 20, 3, device="cuda"), 3, seed=1, step_noise=torch.zeros(10, 2, 20, 3, device="cuda"))
    with pytest.raises(ValueError, match="need a seed"):
        bm.resample(plan, fs, torch.zeros(2, 20, 3, device="cuda"), torch.zeros(2, 20, dtype=torch.bool, device="cuda"), draw=1)
    with pytest.raises(ValueError, match="keys"):
        bm.sample(plan, fs, seed=1, keys=torch.zeros(3, dtype=torch.int64))
    with pytest.raises(ValueError, match="excludes"):
        bm.repair(plan, fs, _clone(bm.sample(plan, fs, seed=1)), seed=1, generator=torch.Generator(device="cuda"))
    traj = synthetic.trajectory(10, 2, seed=1)
    with pytest.raises(ValueError, match="excludes"):
        bm.backmap_coords(traj.ca_full, traj.restype_full, traj.info, seed=1, generator=torch.Generator(device="cuda"))
