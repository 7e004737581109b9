"""GPU tests of latent inpainting (run on the B200 box: pytest -m gpu): the fused step loop of both tiers against the CPU
oracle's restatement (tests/inpaint_oracle.py) under DDPM and DDIM with per-member masks, graph replay, the all-False
identity with a plain pass, the plan's inpainting state and Backmapper.resample.  The reference has no inpainting, so these
results are pinned against the restatement, which is tied to the pinned oracle by the all-False identity."""
import pytest
import torch

from codlad_b200 import synthetic, weights
from tests import inpaint_oracle as I
from tests import parity_utils as P
from tests.test_gpu_ddim import _inputs, _plan

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
def inpaint_cache():
    """Inputs per case, and oracle results per (case, variant, mask), shared by the tests of this module."""
    return {}


# name -> (sampler, respacing, eta)
VARIANTS = {"ddpm10": ("ddpm", "10", 0.0), "ddim50_eta0": ("ddim", "ddim50", 0.0), "ddim50_eta1": ("ddim", "ddim50", 1.0)}
MASKS = ["window", "scattered", "ends", "padded"]


def _case(cache, case):
    key = ("inputs", case)
    if key not in cache:
        inp = _inputs(case)
        inp["valid"] = inp["mask"][inp["frame_of"].long()]
        inp["x0"] = synthetic.latent_noise(tuple(inp["z0"].shape), 2304)     # the normalised latent to keep
        cache[key] = inp
    return cache[key]


def _keep(inp, kind):
    """Per-member masks [NB, L]: a window that moves with the member, scattered rows, the first and last valid residue, or
    every padded row plus the first six."""
    valid = inp["valid"]
    NB, L = valid.shape
    keep = torch.zeros(NB, L, dtype=torch.bool)
    for b in range(NB):
        n = int(valid[b].sum())
        if kind == "window":
            keep[b, 8 + 4 * b:24 + 4 * b] = True
        elif kind == "scattered":
            keep[b] = torch.rand(L, generator=torch.Generator().manual_seed(50 + b)) < 0.3
        elif kind == "ends":
            keep[b, 0] = keep[b, n - 1] = True
        else:
            keep[b, n:] = True
            keep[b, :6] = True
    return keep


def _set_schedule(plan, diff, sampler, eta):
    if sampler == "ddim":
        plan.set_ddim_schedule(diff.timestep_map, diff.ddim_coef_table(eta))
    else:
        plan.set_schedule(diff.timestep_map, diff.coef_table())


def _noise(inp, T, sampler, eta):
    return inp["noises"][:T].cuda().contiguous() if sampler == "ddpm" or eta != 0 else None


def _oracle(sd, inp, cache, case, variant, mask, keep):
    key = (case, variant, mask)
    if key not in cache:
        sampler, spacing, eta = VARIANTS[variant]
        fo = inp["frame_of"].long()
        T = len(I.level_table(spacing)) - 1
        noises = inp["noises"][:T] if sampler == "ddpm" or eta != 0 else None
        cache[key] = I.sample_loop(sd, inp["z0"], inp["X"][fo], inp["cg_z"][fo], inp["mask"][fo], noises, spacing, keep, inp["x0"],
                                   sampler, eta)
    return cache[key]


# Relative-error bars of the free rows, about 3x the worst value measured on a B200 over both cases, all three variants and all
# four masks: fp32 tier 4.9e-7, f16 tier 5.4e-4 (the DDIM bars, which these equal).
BARS = {"fp32": 1.5e-6, "f16": 1.5e-3}


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("case", ["golden", "ragged"])
def test_fused_inpaint_loop_vs_oracle(eng, denoiser, inpaint_cache, case, variant, mask, precision):
    """plan.sample with inpainting on against the oracle: free rows within the bar, kept rows exactly x0, CUDA-graph replay
    bit-identical to eager launches."""
    from codlad_b200.diffusion import create_diffusion
    sd, den = denoiser
    sampler, spacing, eta = VARIANTS[variant]
    inp = _case(inpaint_cache, case)
    keep = _keep(inp, mask)
    ref = _oracle(sd, inp, inpaint_cache, case, variant, mask, keep)
    diff = create_diffusion(spacing)
    plan = _plan(eng, den, inp, precision)
    _set_schedule(plan, diff, sampler, eta)
    plan.set_inpaint(keep.cuda(), inp["x0"].cuda(), diff.inpaint_coef_table())
    nz = _noise(inp, diff.num_timesteps, sampler, eta)
    x = plan.sample(inp["z0"].cuda().clone(), nz, use_graph=False).cpu()
    free = inp["valid"] & ~keep
    err = P.rel_err(x[free], ref[free])
    print(f"inpaint {case} {variant} {mask} {precision}: free rows rel err vs oracle {err:.3e}, kept {int(keep.sum())} rows")
    assert torch.isfinite(x).all()
    assert torch.equal(x[keep], inp["x0"][keep])
    assert err < BARS[precision], err
    xg = plan.sample(inp["z0"].cuda().clone(), nz, use_graph=True)
    assert torch.equal(xg.cpu(), x), "CUDA-graph replay must equal the eager launch sequence bit for bit"


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_marked_padded_rows_leave_valid_rows_alone(eng, denoiser, inpaint_cache, precision):
    """Marking padded rows as kept changes no valid row."""
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    inp = _case(inpaint_cache, "ragged")
    diff = create_diffusion("10")
    plan = _plan(eng, den, inp, precision)
    plan.set_schedule(diff.timestep_map, diff.coef_table())
    nz = _noise(inp, 10, "ddpm", 0.0)
    keep = _keep(inp, "padded")
    res = []
    for k in (keep, keep & inp["valid"]):
        plan.set_inpaint(k.cuda(), inp["x0"].cuda(), diff.inpaint_coef_table())
        res.append(plan.sample(inp["z0"].cuda().clone(), nz).cpu())
    assert torch.equal(res[0][inp["valid"]], res[1][inp["valid"]])


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("variant", ["ddpm10", "ddim50_eta0"])
def test_all_false_keep_is_a_plain_pass(eng, denoiser, inpaint_cache, variant, precision):
    """An all-False keep mask gives a plain pass bit for bit, through the graph."""
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    sampler, spacing, eta = VARIANTS[variant]
    inp = _case(inpaint_cache, "ragged")
    diff = create_diffusion(spacing)
    nz = _noise(inp, diff.num_timesteps, sampler, eta)
    plan = _plan(eng, den, inp, precision)
    _set_schedule(plan, diff, sampler, eta)
    plain = plan.sample(inp["z0"].cuda().clone(), nz).clone()
    plan.set_inpaint(torch.zeros(inp["valid"].shape, dtype=torch.bool, device="cuda"), inp["x0"].cuda(), diff.inpaint_coef_table())
    masked = plan.sample(inp["z0"].cuda().clone(), nz)
    assert torch.equal(masked, plain)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_plan_inpaint_state(eng, denoiser, inpaint_cache, precision):
    """plain -> inpaint -> plain gives the first plain result again; new keep / x0 between two inpaint passes give what a fresh
    plan gives, with one launch more than a plain pass; an inpainting table of another T is refused."""
    from codlad_b200.diffusion import create_diffusion
    _, den = denoiser
    inp = _case(inpaint_cache, "ragged")
    diff = create_diffusion("10")
    q = diff.inpaint_coef_table()
    nz = _noise(inp, 10, "ddpm", 0.0)
    z0 = inp["z0"].cuda()
    k1, k2 = _keep(inp, "window").cuda(), _keep(inp, "scattered").cuda()
    x01, x02 = inp["x0"].cuda(), synthetic.latent_noise(tuple(inp["z0"].shape), 2305).cuda()
    plan = _plan(eng, den, inp, precision)
    plan.set_schedule(diff.timestep_map, diff.coef_table())
    first = plan.sample(z0.clone(), nz).clone()
    l0 = plan.launches
    plan.sample(z0.clone(), nz)
    plain_launches = plan.launches - l0
    plan.set_inpaint(k1, x01, q)
    a = plan.sample(z0.clone(), nz).clone()
    plan.set_inpaint(k2, x02, q)
    l0 = plan.launches
    b = plan.sample(z0.clone(), nz).clone()
    assert plan.launches - l0 == plain_launches + 1
    plan.clear_inpaint()
    again = plan.sample(z0.clone(), nz).clone()
    fresh = _plan(eng, den, inp, precision)
    fresh.set_schedule(diff.timestep_map, diff.coef_table())
    fresh.set_inpaint(k2, x02, q)
    want = fresh.sample(z0.clone(), nz)
    torch.cuda.synchronize()
    assert torch.equal(first, again)
    assert torch.equal(b, want)
    assert not torch.equal(a, b) and not torch.equal(a, first)
    plan.set_inpaint(k1, x01, create_diffusion("25").inpaint_coef_table())
    with pytest.raises(RuntimeError, match="inpainting table"):
        plan.sample(z0.clone(), nz)


def _backmapper_case():
    prot = synthetic.make_protein(120, 1, seed=1011)
    from codlad_b200 import sampler
    fs = sampler.frames_from_batch(synthetic.collate(prot), prot.info, 4)
    return fs, synthetic.latent_noise((4, 120, 3), 2011), synthetic.latent_noise((4, 120, 3), 2012), synthetic.latent_noise((25, 4, 120, 3), 2013)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_backmapper_resample(precision):
    """Backmapper.resample, 25 DDPM steps, 4 members of a 120-residue protein: an all-True mask reproduces the earlier pass's
    idx, ic_recon and xyz; with a partial mask kept rows keep latent and VQ index while free rows change; the previous call's
    own latent buffer gives what a clone gives; sample() after resample() is a plain pass again."""
    from codlad_b200 import sampler
    fs, z1, z2, sn = _backmapper_case()
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=25,
                            precision=precision)
    plan = bm.upload(fs)
    out = bm.sample(plan, fs, z1, sn)
    first = {k: v.clone() for k, v in out.items()}
    same = bm.resample(plan, fs, first["latent"], torch.ones(4, 120, dtype=torch.bool, device="cuda"), z=z2, step_noise=sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(same[k], first[k]), k
    keep = torch.zeros(4, 120, dtype=torch.bool)
    keep[:, 30:70] = True
    keep[2, :5] = True
    keep = keep.cuda()
    part = {k: v.clone() for k, v in bm.resample(plan, fs, first["latent"], keep, z=z2, step_noise=sn).items()}
    assert torch.equal(part["latent"][keep], first["latent"][keep])
    assert torch.equal(part["idx"][keep], first["idx"][keep])
    assert not torch.equal(part["latent"][~keep], first["latent"][~keep])
    bm.sample(plan, fs, z1, sn)                                 # the plan's latent buffer holds the first pass again
    aliased = bm.resample(plan, fs, bm._bufs[id(plan)][0], keep, z=z2, step_noise=sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(aliased[k], part[k]), k
    plain = bm.sample(plan, fs, z1, sn)
    for k in ("latent", "idx", "ic_recon", "xyz"):
        assert torch.equal(plain[k], first[k]), k


def test_backmapper_resample_ddim_eta0_needs_no_noise():
    """DDIM at eta = 0: resample allocates no step-noise buffer and matches the plan-level inpainting loop."""
    from codlad_b200 import engine, sampler
    fs, z1, z2, _ = _backmapper_case()
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=25,
                            precision="f16", sampler="ddim", eta=0.0)
    plan = bm.upload(fs)
    lat = bm.sample(plan, fs, z1)["latent"].clone()
    keep = torch.zeros(4, 120, dtype=torch.bool, device="cuda")
    keep[:, ::3] = True
    out = bm.resample(plan, fs, lat, keep, z=z2)
    assert bm._bufs[id(plan)][1] is None
    assert torch.equal(out["latent"][keep], lat[keep])
    ref = engine.Plan(bm.denoiser, fs.F, fs.NB, fs.L, "f16")
    ref.set_frames(fs.X, fs.lengths, fs.cg_z, fs.frame_of)
    ref.set_ddim_schedule(bm.diffusion.timestep_map, bm.diffusion.ddim_coef_table(0.0))
    ref.set_inpaint(keep, lat, bm.diffusion.inpaint_coef_table())
    assert torch.equal(ref.sample(z2.cuda().clone(), None, use_graph=False), out["latent"])


def test_resample_rejects_bad_arguments():
    from codlad_b200 import sampler
    fs, z1, _, _ = _backmapper_case()
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=10,
                            precision="fp32")
    plan = bm.upload(fs)
    lat = bm.sample(plan, fs, z1)["latent"].clone()
    keep = torch.zeros(4, 120, dtype=torch.bool, device="cuda")
    for bad_lat, bad_keep in ((lat, keep.to(torch.uint8)), (lat, keep[:, :100]), (lat, keep.cpu()), (lat.double(), keep),
                              (lat[:, :100], keep), (lat.cpu(), keep), (lat[..., :2], keep)):
        with pytest.raises(ValueError):
            bm.resample(plan, fs, bad_lat, bad_keep)
    with pytest.raises(ValueError):
        plan.set_inpaint(keep, lat, bm.diffusion.inpaint_coef_table()[:, :1])
