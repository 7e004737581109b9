"""CPU: the DDIM coefficient rows the CUDA update consumes, the oracle's restatement of IDDPM's ddim_sample (tied to the
reference-pinned DDPM tables through the eta = 1 identity), and the argument checks that run before any CUDA call."""
import numpy as np
import pytest
import torch

from codlad_b200.diffusion import create_diffusion
from oracle import restate as R
from tests import ddim_oracle as D

SPACINGS = ["1", "10", "25", "100", "1000", "ddim25"]


@pytest.mark.parametrize("spacing", SPACINGS)
@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
def test_ddim_coef_table_matches_float64(spacing, eta):
    d = create_diffusion(spacing)
    c = d.ddim_coef_table(eta)
    T = d.num_timesteps
    assert c.shape == (T, 8) and c.dtype == np.float32
    assert np.isfinite(c).all()
    ac = np.cumprod(1.0 - d.betas)
    ac_prev = np.append(1.0, ac[:-1])
    sigma = eta * np.sqrt((1 - ac_prev) / (1 - ac)) * np.sqrt(1 - ac / ac_prev)
    want = np.zeros((T, 8))
    want[:, 0] = np.sqrt(1 / ac)
    want[:, 1] = np.sqrt(1 / ac - 1)
    want[:, 2] = np.sqrt(ac_prev)
    want[:, 3] = np.sqrt(np.maximum(0.0, 1 - ac_prev - sigma ** 2))
    want[1:, 4] = sigma[1:]
    assert np.array_equal(c, want.astype(np.float32))                 # one rounding of the float64 values
    assert c[0, 4] == 0 and c[0, 3] == 0 and c[0, 2] == 1
    if eta == 0:
        assert (c[:, 4] == 0).all()
    else:
        assert (c[1:, 4] > 0).all()
    assert (c[:, 5:] == 0).all()


@pytest.mark.parametrize("spacing", ["10", "100", "ddim50"])
def test_oracle_schedule_matches_spaced_diffusion(spacing):
    d = create_diffusion(spacing)
    s = D.schedule(spacing)
    assert np.array_equal(s["timestep_map"], np.array(d.timestep_map))
    np.testing.assert_allclose(s["alphas_cumprod"], d.alphas_cumprod, rtol=1e-15, atol=0)
    np.testing.assert_allclose(s["alphas_cumprod_prev"], d.alphas_cumprod_prev, rtol=1e-15, atol=0)
    if not spacing.startswith("ddim"):                                 # the same tables as the reference-pinned oracle
        pinned = R.respaced_schedule(int(spacing))
        for k in ("timestep_map", "betas", "sqrt_recip_ac", "sqrt_recipm1_ac"):
            assert np.array_equal(s[k], pinned[k]), k


@pytest.mark.parametrize("spacing", ["10", "100", "ddim25"])
def test_ddim_at_eta_one_is_the_ddpm_posterior(spacing):
    """At eta = 1, sigma^2 is the DDPM posterior variance and the DDIM mean is the posterior mean q(x_{t-1} | x_t, x0_hat):
    the oracle's ddim_terms (float64) against q_posterior_mean_variance's tables of SpacedDiffusion, every step."""
    d = create_diffusion(spacing)
    s = D.schedule(spacing)
    g = torch.Generator().manual_seed(3)
    for step in range(d.num_timesteps):
        x = torch.randn(2, 17, 3, generator=g, dtype=torch.float64)
        eps = torch.randn(2, 17, 3, generator=g, dtype=torch.float64)
        x0, mean, sigma = D.ddim_terms(x, eps, step, s, 1.0)
        post_mean = d.posterior_mean_coef1[step] * x0 + d.posterior_mean_coef2[step] * x
        assert float((mean - post_mean).abs().max()) < 1e-12, step
        assert abs(float(sigma) ** 2 - d.posterior_variance[step]) < 1e-12, step


def test_oracle_ddim_update_fp32_follows_the_table_rows():
    """The fp32 restatement (IDDPM's order, fp32 tables) and the device formula on the fp32-rounded rows agree closely."""
    d = create_diffusion("ddim50")
    s = D.schedule("ddim50")
    g = torch.Generator().manual_seed(4)
    for eta in (0.0, 1.0):
        c = torch.from_numpy(d.ddim_coef_table(eta))
        for step in (0, 1, 25, 49):
            x, out, z = (torch.randn(3, 40, k, generator=g) for k in (3, 6, 3))
            got = D.ddim_update(x, out, step, z, s, eta)
            r = c[step]
            x0 = r[0] * x - r[1] * out[..., :3]
            want = r[2] * x0 + r[3] * ((r[0] * x - x0) / r[1]) + r[4] * z
            assert torch.allclose(got, want, rtol=1e-5, atol=1e-5), (eta, step)
    x, out = torch.randn(1, 8, 3, generator=g), torch.randn(1, 8, 6, generator=g)
    assert torch.equal(D.ddim_update(x, out, 7, None, s, 0.0), D.ddim_update(x, out, 7, torch.randn(1, 8, 3, generator=g), s, 0.0))


def test_ddim_unsupported_arguments_raise_before_cuda():
    d = create_diffusion("10")
    model = lambda x, t, **kw: torch.zeros(*x.shape[:-1], 6)
    for kw in (dict(clip_denoised=True), dict(clip_denoised=False, cond_fn=lambda *a, **k: 0),
               dict(clip_denoised=False, denoised_fn=lambda v: v)):
        with pytest.raises(NotImplementedError):
            d.ddim_sample_loop(model, (1, 4, 3), **kw)
        with pytest.raises(NotImplementedError):
            next(iter(d.ddim_sample_loop_progressive(model, (1, 4, 3), **kw)))
        with pytest.raises(NotImplementedError):
            d.ddim_sample(model, torch.zeros(1, 4, 3), torch.zeros(1, dtype=torch.int64), **kw)
    with pytest.raises(NotImplementedError):
        d.ddim_sample_loop(model, (1, 4, 3))                           # IDDPM's default clip_denoised=True


def test_backmapper_rejects_unknown_sampler():
    from codlad_b200 import sampler, weights
    with pytest.raises(ValueError):
        sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), sampler="plms")
    with pytest.raises(ValueError):
        sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), eta=0.5)
