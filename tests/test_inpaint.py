"""CPU: the inpainting level table the CUDA overwrite consumes, and the oracle's restatement of latent inpainting, tied to
the pinned DDPM oracle and to the DDIM oracle by the all-False identity (no kept row: the plain loop exactly) and checked at
the other extreme (every row kept: x0 exactly)."""
import numpy as np
import pytest
import torch

from codlad_b200 import synthetic, weights
from codlad_b200.diffusion import create_diffusion
from oracle import restate as R
from tests import ddim_oracle as D
from tests import inpaint_oracle as I


@pytest.mark.parametrize("spacing", ["1", "10", "25", "100", "1000", "ddim25", "ddim50"])
def test_inpaint_coef_table_matches_float64(spacing):
    d = create_diffusion(spacing)
    q = d.inpaint_coef_table()
    T = d.num_timesteps
    assert q.shape == (T + 1, 2) and q.dtype == np.float32
    ac = np.cumprod(1.0 - d.betas)
    level = np.append(np.append(1.0, ac[:-1]), ac[-1])
    want = np.stack([np.sqrt(level), np.sqrt(1.0 - level)], axis=1)
    assert np.array_equal(q, want.astype(np.float32))                   # one rounding of the float64 values
    assert q[0, 0] == 1.0 and q[0, 1] == 0.0                            # kept rows end at x0 exactly
    assert (np.diff(q[:, 0]) <= 0).all() and (np.diff(q[:, 1]) >= 0).all()     # noisier level at every earlier step
    assert np.array_equal(I.level_table(spacing).numpy(), q)


@pytest.fixture
def one_thread():
    """The identities below compare two CPU loops bit for bit; a matrix product may sum in another order when the library
    picks another thread count between calls, so both loops run on one thread."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _case(L=24, B=2, seed=77):
    prot = synthetic.make_protein(L, 1, seed=seed)
    X = prot.ca_full[:, 1:-1].expand(B, -1, -1).contiguous()
    cg_z = prot.restype_full[1:-1][None].expand(B, -1).contiguous()
    mask = torch.ones(B, L, dtype=torch.bool)
    mask[1, L - 5:] = False                                             # a padded tail on the second member
    return dict(sd=weights.init_denoiser_state(0), X=X, cg_z=cg_z, mask=mask, z=synthetic.latent_noise((B, L, 3), seed + 1),
                noises=synthetic.latent_noise((10, B, L, 3), seed + 2), x0=synthetic.latent_noise((B, L, 3), seed + 3))


def test_all_false_keep_is_the_plain_ddpm_loop(one_thread):
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    got = I.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], c["noises"], "10", keep, c["x0"], "ddpm")
    want = R.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], c["noises"], R.respaced_schedule(10))
    assert torch.equal(got, want)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_all_false_keep_is_the_plain_ddim_loop(one_thread, eta):
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    noises = c["noises"] if eta != 0 else None
    got = I.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], noises, "10", keep, c["x0"], "ddim", eta)
    want = D.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], noises, D.schedule("10"), eta)
    assert torch.equal(got, want)


@pytest.mark.parametrize("sampler,eta", [("ddpm", 0.0), ("ddim", 0.0), ("ddim", 1.0)])
def test_all_true_keep_returns_x0(sampler, eta):
    c = _case()
    keep = torch.ones(c["mask"].shape, dtype=torch.bool)
    noises = c["noises"] if sampler == "ddpm" or eta != 0 else None
    got = I.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], noises, "10", keep, c["x0"], sampler, eta)
    assert torch.equal(got, c["x0"])


def test_partial_keep_conditions_the_free_rows():
    """Kept rows end at x0; the free rows differ from the plain loop's (they are conditioned on the kept ones)."""
    c = _case()
    keep = torch.zeros(c["mask"].shape, dtype=torch.bool)
    keep[:, 5:12] = True
    got = I.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], None, "10", keep, c["x0"], "ddim", 0.0)
    plain = D.sample_loop(c["sd"], c["z"], c["X"], c["cg_z"], c["mask"], None, D.schedule("10"), 0.0)
    assert torch.equal(got[keep], c["x0"][keep])
    free = ~keep & c["mask"]
    assert not torch.equal(got[free], plain[free])
