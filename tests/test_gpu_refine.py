"""GPU tests of partial-noise refinement (run on the B200 box: pytest -m gpu): a refinement pass of the fused step loop against a
plain pass on the truncated schedule (bit for bit) and against the CPU restatement (tests/refine_oracle.py), graph replay across
starts, plan state after refinement, the C side's refusals, Backmapper.residue_motion, Backmapper.backmap_trajectory against the
hand-written sequence of passes, and the warm start's coherence.  The reference has no refinement, so these results are pinned
against the restatement, which is tied to the pinned oracle (tests/test_refine.py)."""
import math

import pytest
import torch

from codlad_b200 import synthetic, weights
from oracle import restate as R
from tests import parity_utils as P
from tests import refine_oracle as O
from tests.test_gpu_ddim import _plan
from tests.test_gpu_inpaint import BARS, VARIANTS, _case, _keep, _noise, _set_schedule

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


@pytest.fixture(scope="module")
def eng():
    from codlad_b200 import engine
    return engine


@pytest.fixture(scope="module")
def denoiser(eng):
    sd = weights.init_denoiser_state(0)
    return sd, eng.DenoiserEngine(sd, 64)


@pytest.fixture(scope="module")
def cache():
    return {}


def _starts(T):
    return {"1": 1, "half": T // 2, "T": T}


def _level(q, s, x0, z):
    """level_s(x0, z) in fp32 on the host: two rounded products and one rounded sum."""
    q = torch.as_tensor(q)
    return q[s, 0] * x0 + q[s, 1] * z


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("start", ["1", "half", "T"])
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("case", ["golden", "ragged"])
def test_refine_is_a_plain_pass_on_the_truncated_schedule(eng, denoiser, cache, case, variant, start, precision):
    """A start of s steps with no kept row equals a plain pass on a plan loaded with the first s rows of the same schedule, started
    from level_s(x0, z) computed on the host, with the same noise slices: bit for bit, through the graph."""
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    sampler, spacing, eta = VARIANTS[variant]
    inp = _case(cache, case)
    diff = create_diffusion(spacing)
    T = diff.num_timesteps
    s = _starts(T)[start]
    q = diff.inpaint_coef_table()
    nz = _noise(inp, T, sampler, eta)
    plan = _plan(eng, den, inp, precision)
    _set_schedule(plan, diff, sampler, eta)
    plan.set_inpaint(torch.zeros(inp["valid"].shape, dtype=torch.bool, device="cuda"), inp["x0"].cuda(), q)
    plan.set_start(s)
    l0 = plan.launches
    got = plan.sample(inp["z0"].cuda().clone(), nz)
    assert plan.launches - l0 == 16 * s + 1
    short = _plan(eng, den, inp, precision)
    coef = diff.ddim_coef_table(eta) if sampler == "ddim" else diff.coef_table()
    (short.set_ddim_schedule if sampler == "ddim" else short.set_schedule)(diff.timestep_map[:s], coef[:s])
    want = short.sample(_level(q, s, inp["x0"], inp["z0"]).cuda(), None if nz is None else nz[:s].contiguous())
    assert torch.equal(got, want)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("mask", ["none", "window", "padded"])
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("case", ["golden", "ragged"])
def test_refine_vs_oracle(eng, denoiser, cache, case, variant, mask, precision):
    """Half-strength refinement against the oracle: free rows within the inpainting bars, kept rows exactly x0."""
    from codlad_b200.diffusion import create_diffusion
    sd, den = denoiser
    sampler, spacing, eta = VARIANTS[variant]
    inp = _case(cache, case)
    keep = torch.zeros(inp["valid"].shape, dtype=torch.bool) if mask == "none" else _keep(inp, mask)
    diff = create_diffusion(spacing)
    T = diff.num_timesteps
    s = T // 2
    key = ("refine", case, variant, mask)
    if key not in cache:
        fo = inp["frame_of"].long()
        noises = inp["noises"][:T] if sampler == "ddpm" or eta != 0 else None
        cache[key] = O.sample_loop(sd, inp["z0"], inp["X"][fo], inp["cg_z"][fo], inp["mask"][fo], noises, spacing, s, keep, inp["x0"],
                                   sampler, eta)
    ref = cache[key]
    plan = _plan(eng, den, inp, precision)
    _set_schedule(plan, diff, sampler, eta)
    plan.set_inpaint(keep.cuda(), inp["x0"].cuda(), diff.inpaint_coef_table())
    plan.set_start(s)
    x = plan.sample(inp["z0"].cuda().clone(), _noise(inp, T, sampler, eta)).cpu()
    free = inp["valid"] & ~keep
    err = P.rel_err(x[free], ref[free])
    print(f"refine {case} {variant} {mask} {precision} steps {s}/{T}: free rows rel err vs oracle {err:.3e}, kept {int(keep.sum())} rows")
    assert torch.isfinite(x).all()
    assert torch.equal(x[keep], inp["x0"][keep])
    assert err < BARS[precision], err


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_graph_replay_across_starts(eng, denoiser, cache, precision):
    """Graph replay equals eager launches while one plan switches starts s1 -> s2 -> s1 (each switch re-captures), and the two s1
    passes agree; a start of 0 is the full inpainting pass again."""
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    inp = _case(cache, "ragged")
    diff = create_diffusion("10")
    nz = _noise(inp, 10, "ddpm", 0.0)
    keep = _keep(inp, "window").cuda()
    plan = _plan(eng, den, inp, precision)
    plan.set_schedule(diff.timestep_map, diff.coef_table())
    plan.set_inpaint(keep, inp["x0"].cuda(), diff.inpaint_coef_table())
    z0 = inp["z0"].cuda()
    full = plan.sample(z0.clone(), nz).clone()
    res = []
    for s in (3, 7, 3):
        plan.set_start(s)
        g = plan.sample(z0.clone(), nz, use_graph=True).clone()
        e = plan.sample(z0.clone(), nz, use_graph=False).clone()
        assert torch.equal(g, e), f"graph != eager at start {s}"
        res.append(g)
    assert torch.equal(res[0], res[2]) and not torch.equal(res[0], res[1])
    plan.set_start(0)
    assert torch.equal(plan.sample(z0.clone(), nz), full)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_c_side_refusals(eng, denoiser, cache, precision):
    from codlad_b200 import _native as N
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    inp = _case(cache, "ragged")
    diff = create_diffusion("10")
    nz = _noise(inp, 10, "ddpm", 0.0)
    plan = _plan(eng, den, inp, precision)
    plan.set_schedule(diff.timestep_map, diff.coef_table())
    plan.set_inpaint(torch.zeros(inp["valid"].shape, dtype=torch.bool, device="cuda"), inp["x0"].cuda(), diff.inpaint_coef_table())
    plan.set_start(11)
    with pytest.raises(RuntimeError, match="exceeds the schedule"):
        plan.sample(inp["z0"].cuda().clone(), nz)
    plan.clear_inpaint()
    plan.set_start(4)
    with pytest.raises(RuntimeError, match="cb2_plan_set_inpaint"):
        plan.sample(inp["z0"].cuda().clone(), nz)
    assert N.lib().cb2_plan_set_start(plan.handle, -1, None) != 0
    assert b"steps must be >= 0" in N.lib().cb2_last_error()
    with pytest.raises(ValueError):
        plan.set_start(-1)
    plan.set_start(0)
    plan.sample(inp["z0"].cuda().clone(), nz)                            # a plain pass again


# ---- Backmapper -------------------------------------------------------------------------------------------------------------------
def _bm(precision="f16", steps=10, sampler="ddpm", eta=0.0):
    from codlad_b200 import sampler as S
    return S.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=steps,
                        precision=precision, sampler=sampler, eta=eta)


def _protein_fs(L=60, NB=3, seed=1201):
    from codlad_b200 import sampler as S
    prot = synthetic.make_protein(L, 1, seed=seed)
    return S.frames_from_batch(synthetic.collate(prot), prot.info, NB)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_backmapper_refine_leaves_sample_and_resample_alone(precision):
    """On a fresh plan: sample() and resample(); then refine() with and without a keep mask; then sample() and resample() again give
    the first results bit for bit.  refine(keep) keeps the kept residues' latent and VQ index.  DDPM-10, 3 members."""
    fs = _protein_fs()
    bm = _bm(precision)
    z1, z2 = synthetic.latent_noise((3, 60, 3), 31), synthetic.latent_noise((3, 60, 3), 32)
    sn = synthetic.latent_noise((10, 3, 60, 3), 33)
    keep = torch.zeros(3, 60, dtype=torch.bool, device="cuda")
    keep[:, 10:30] = True
    plan = bm.upload(fs)
    first = {k: v.clone() for k, v in bm.sample(plan, fs, z1, sn).items()}
    res1 = {k: v.clone() for k, v in bm.resample(plan, fs, first["latent"], keep, z=z2, step_noise=sn).items()}
    ref = bm.refine(plan, fs, first["latent"], 4, z=z2, step_noise=sn)
    assert not torch.equal(ref["latent"], first["latent"])
    part = bm.refine(plan, fs, first["latent"], 4, keep=keep, z=z2, step_noise=sn)
    assert torch.equal(part["latent"][keep], first["latent"][keep]) and torch.equal(part["idx"][keep], first["idx"][keep])
    again = bm.sample(plan, fs, z1, sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(again[k], first[k]), k
    res2 = bm.resample(plan, fs, first["latent"], keep, z=z2, step_noise=sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(res2[k], res1[k]), k


def test_backmapper_refine_ddim_eta0_needs_no_noise():
    fs = _protein_fs()
    bm = _bm("f16", 25, "ddim", 0.0)
    plan = bm.upload(fs)
    lat = bm.sample(plan, fs, synthetic.latent_noise((3, 60, 3), 41))["latent"]
    out = bm.refine(plan, fs, lat, 6, z=synthetic.latent_noise((3, 60, 3), 42))
    assert bm._bufs[id(plan)][1] is None
    assert torch.isfinite(out["latent"]).all()


def test_residue_motion():
    """Rigid-body moves of whole residues give 0; a planted side-chain move gives the oracle's float64 Kabsch RMSD of that residue; padded
    rows give NaN.  Two proteins of 50 and 41 residues padded to 50, two members on each."""
    from codlad_b200 import sampler as S
    p1, p2 = synthetic.make_protein(50, 1, seed=51), synthetic.make_protein(41, 1, seed=52)
    fs = S.frames_from_batch(synthetic.collate_many([p1, p2]), [p1.info, p2.info], 2)
    bm = _bm("f16")
    plan = bm.upload(fs)
    xyz = bm.sample(plan, fs, generator=torch.Generator(device="cuda").manual_seed(5))["xyz"].clone()
    atoms, counts, rows = S.residue_atom_ranges(fs)
    starts = torch.cumsum(counts, 0) - counts
    g = torch.Generator().manual_seed(7)
    moved = xyz.cpu().double()
    for r in range(rows.numel()):                          # every residue: its own rotation and translation
        idx = atoms[starts[r]:starts[r] + counts[r]]
        qr, _ = torch.linalg.qr(torch.randn(3, 3, generator=g, dtype=torch.float64))
        qr = qr * torch.sign(torch.det(qr))
        moved[idx] = moved[idx] @ qr.T + 10.0 * torch.randn(3, generator=g, dtype=torch.float64)
    rigid = bm.residue_motion(fs, xyz, moved.float().cuda()).cpu()
    valid = fs.lengths.long()[fs.frame_of.long()][:, None] > torch.arange(fs.L)[None]
    assert rigid.dtype == torch.float64 and rigid.shape == (fs.NB, fs.L)
    assert torch.isnan(rigid[~valid]).all() and int((~valid).sum()) == 2 * 9
    assert float(rigid[valid].abs().max()) < 1e-4, float(rigid[valid].abs().max())
    planted = xyz.clone()
    r = int(torch.nonzero(counts >= 7)[3])                 # a residue with a side chain
    idx = atoms[starts[r]:starts[r] + counts[r]]
    planted[idx[-1]] += torch.tensor([0.9, -0.4, 0.3], device="cuda")
    planted[idx[-2]] += torch.tensor([-0.2, 0.5, 0.0], device="cuda")
    got = bm.residue_motion(fs, xyz, planted).cpu().flatten()
    want = R.superposed_rmsd(xyz[idx].cpu().numpy(), planted[idx].cpu().numpy())
    print(f"residue_motion: rigid max {float(rigid[valid].abs().max()):.2e}, planted {float(got[rows[r]]):.6f} vs {want:.6f}")
    assert want > 0.1 and math.isclose(float(got[rows[r]]), want, rel_tol=1e-5, abs_tol=1e-6)
    others = torch.ones(fs.NB * fs.L, dtype=torch.bool)
    others[rows[r]] = False
    assert float(got[others & valid.flatten()].abs().max()) < 1e-3


def _trajectory(n=7, L=40, seed=61):
    prot = synthetic.trajectory(L, n, seed=seed)
    return [synthetic.collate(prot, [f]) for f in range(n)], prot.info


@pytest.mark.parametrize("chunks", [1, 3])
def test_backmap_trajectory_is_the_sequence_of_passes(chunks):
    """backmap_trajectory equals sample() on the first frame of every chunk, then refine() of each member from its own latent on the
    chunk's next frame (the last frame repeated once a chunk has ended), on one plan with one generator: bit for bit."""
    from codlad_b200 import batching
    from codlad_b200 import sampler as S
    batches, info = _trajectory()
    E, steps = 2, 3
    bm = _bm("f16")
    got = bm.backmap_trajectory(batches, info, num_ensemble=E, steps=steps, chunks=chunks,
                                generator=torch.Generator(device="cuda").manual_seed(99))
    assert got.shape == (7, E, int(info[0].numel()), 3) and got.dtype == torch.float32 and not got.is_cuda
    runs = S.trajectory_chunks(7, chunks)
    gen = torch.Generator(device="cuda").manual_seed(99)
    want = torch.empty_like(got)
    plans = set()
    for p in range(max(n for _, n in runs)):
        frames = [s + min(p, n - 1) for s, n in runs]
        fs = S.frames_from_batch(batching.merge_batches([batches[f] for f in frames]), info, E)
        plan = bm.upload(fs)
        plans.add(id(plan))
        out = bm.sample(plan, fs, generator=gen) if p == 0 else bm.refine(plan, fs, out["latent"], steps, generator=gen)
        xyz = out["xyz"].view(E, chunks, -1, 3).cpu()
        for c, (s, n) in enumerate(runs):
            if p < n:
                want[s + p] = xyz[:, c]
    assert len(plans) == 1
    assert torch.equal(got, want)


def test_warm_start_keeps_the_vq_indices():
    """Mechanics of coherence: DDIM-25, eta = 0, refinement of one step from the previous frame's latent keeps at least 90 % of
    the VQ indices between consecutive frames; independent samples of the same frames keep far fewer.  Says nothing about sample
    quality (random-init weights)."""
    from codlad_b200 import sampler as S
    batches, info = _trajectory(6, 60, seed=71)
    bm = _bm("f16", 25, "ddim", 0.0)
    gen = torch.Generator(device="cuda").manual_seed(3)
    warm, cold = [], []
    for f, batch in enumerate(batches):
        fs = S.frames_from_batch(batch, info, 4)
        plan = bm.upload(fs)
        if f == 0:
            out = bm.sample(plan, fs, generator=gen)
            w = c = out["idx"].clone()
        else:
            c = bm.sample(plan, fs, generator=gen)["idx"].clone()          # an independent sample of this frame
            out = bm.refine(plan, fs, lat, 1, generator=gen)
            w = out["idx"].clone()
            warm.append(float((w == prev_w).float().mean()))
            cold.append(float((c == prev_c).float().mean()))
        lat = out["latent"].clone()
        prev_w, prev_c = w, c
    print(f"VQ indices kept between consecutive frames: warm start {min(warm):.3f}..{max(warm):.3f}, independent "
          f"{min(cold):.3f}..{max(cold):.3f}")
    assert min(warm) >= 0.9
    assert max(cold) < 0.5
