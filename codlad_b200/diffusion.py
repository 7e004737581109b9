"""Diffusion process objects with the reference's call surface
(`diffusion_and_flow/__init__.py:10-60`, `respace.py`, `gaussian_diffusion.py`), sampling side.

Coefficient tables are float64 numpy exactly as the reference builds them (they are tiny, host-side,
computed once).  The step loop itself is CUDA:
  * when the model is a `codlad_b200.latent_model` denoiser, `p_sample_loop` hands the whole loop
    (T denoiser forwards + T fused p_sample updates) to `cb2_plan_sample` as one CUDA graph;
  * any other callable goes through a generic loop whose update is the `cb2_p_sample` kernel.
`ddim_sample_loop` (IDDPM's DDIM sampler, which the reference does not ship) takes the same two routes with the DDIM
update (`cb2_plan_set_ddim_schedule` / `cb2_ddim_sample`).  `inpaint_coef_table` feeds latent inpainting on a plan
(`cb2_plan_set_inpaint`, `sampler.Backmapper.resample`).
`training_losses` (config 5, "next" row f-1 of SURVEY.md section 8) is not implemented yet.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _native as N


def get_named_beta_schedule(schedule_name: str, num_diffusion_timesteps: int) -> np.ndarray:
    """gaussian_diffusion.py:104-129."""
    if schedule_name == "linear":
        scale = 1000 / num_diffusion_timesteps
        return np.linspace(scale * 0.0001, scale * 0.02, num_diffusion_timesteps, dtype=np.float64)
    if schedule_name == "squaredcos_cap_v2":
        f = lambda t: math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2
        n = num_diffusion_timesteps
        return np.array([min(1 - f((i + 1) / n) / f(i / n), 0.999) for i in range(n)])
    raise NotImplementedError(f"unknown beta schedule: {schedule_name}")


def space_timesteps(num_timesteps: int, section_counts) -> set:
    """respace.py:12-62."""
    if isinstance(section_counts, str):
        if section_counts.startswith("ddim"):
            want = int(section_counts[4:])
            for stride in range(1, num_timesteps):
                if len(range(0, num_timesteps, stride)) == want:
                    return set(range(0, num_timesteps, stride))
            raise ValueError(f"cannot create exactly {num_timesteps} steps with an integer stride")
        section_counts = [int(x) for x in section_counts.split(",")]
    per, extra = divmod(num_timesteps, len(section_counts))
    start, steps = 0, []
    for i, count in enumerate(section_counts):
        size = per + (1 if i < extra else 0)
        if size < count:
            raise ValueError(f"cannot divide section of {size} steps into {count}")
        stride = 1 if count <= 1 else (size - 1) / (count - 1)
        cur = 0.0
        for _ in range(count):
            steps.append(start + round(cur))
            cur += stride
        start += size
    return set(steps)


class SpacedDiffusion:
    """Respaced DDPM with epsilon prediction and learned-range variance (the configuration
    create_diffusion builds for test.py:298-303).  Attribute names follow the reference."""

    def __init__(self, use_timesteps, betas, learn_sigma=True, predict_xstart=False, sigma_small=False, self_condition=False,
                 loss_type="mse"):
        if predict_xstart or not learn_sigma or self_condition:
            raise NotImplementedError("codlad_b200 implements the sampling configuration of the reference's inference "
                                      "script: epsilon prediction, learn_sigma=True, no self-conditioning")
        self.use_timesteps = set(use_timesteps)
        self.loss_type = loss_type
        base = np.array(betas, dtype=np.float64)
        self.original_num_steps = len(base)
        base_ac = np.cumprod(1.0 - base, axis=0)
        last, new_betas, self.timestep_map = 1.0, [], []
        for i, ac in enumerate(base_ac):
            if i in self.use_timesteps:
                new_betas.append(1 - ac / last)
                last = ac
                self.timestep_map.append(i)
        b = self.betas = np.array(new_betas, dtype=np.float64)
        assert (b > 0).all() and (b <= 1).all()
        self.num_timesteps = int(b.shape[0])
        self.self_condition = False
        ac = self.alphas_cumprod = np.cumprod(1.0 - b, axis=0)
        self.alphas_cumprod_prev = np.append(1.0, ac[:-1])
        self.alphas_cumprod_next = np.append(ac[1:], 0.0)
        self.sqrt_alphas_cumprod = np.sqrt(ac)
        self.sqrt_one_minus_alphas_cumprod = np.sqrt(1.0 - ac)
        self.sqrt_recip_alphas_cumprod = np.sqrt(1.0 / ac)
        self.sqrt_recipm1_alphas_cumprod = np.sqrt(1.0 / ac - 1)
        self.posterior_variance = b * (1.0 - self.alphas_cumprod_prev) / (1.0 - ac)
        self.posterior_log_variance_clipped = (
            np.log(np.append(self.posterior_variance[1], self.posterior_variance[1:])) if len(b) > 1 else np.array([]))
        self.posterior_mean_coef1 = b * np.sqrt(self.alphas_cumprod_prev) / (1.0 - ac)
        self.posterior_mean_coef2 = (1.0 - self.alphas_cumprod_prev) * np.sqrt(1.0 - b) / (1.0 - ac)
        self._coef_dev = {}

    # -- tables for the CUDA side --------------------------------------------------------------
    def coef_table(self) -> np.ndarray:
        """[T, 8] fp32 rows consumed by cb2_plan_set_schedule / cb2_p_sample
        (.float() of the float64 tables, as gaussian_diffusion.py:737 does)."""
        T = self.num_timesteps
        c = np.zeros((T, 8), dtype=np.float32)
        c[:, 0] = self.posterior_log_variance_clipped
        c[:, 1] = np.log(self.betas)
        c[:, 2] = self.sqrt_recip_alphas_cumprod
        c[:, 3] = self.sqrt_recipm1_alphas_cumprod
        c[:, 4] = self.posterior_mean_coef1
        c[:, 5] = self.posterior_mean_coef2
        c[:, 6] = (np.arange(T) != 0).astype(np.float32)
        return c

    def ddim_coef_table(self, eta: float = 0.0) -> np.ndarray:
        """[T, 8] fp32 rows consumed by cb2_plan_set_ddim_schedule / cb2_ddim_sample, computed in float64 and rounded once:
        {sqrt(1/acp), sqrt(1/acp - 1), sqrt(acp_prev), sqrt(max(0, 1 - acp_prev - sigma^2)), sigma * (step != 0), 0, 0, 0} with
        sigma = eta sqrt((1 - acp_prev) / (1 - acp)) sqrt(1 - acp / acp_prev) (IDDPM gaussian_diffusion.py ddim_sample).  The max
        keeps rounding near eta = 1 from turning a tiny argument into a NaN."""
        ac, ac_prev = self.alphas_cumprod, self.alphas_cumprod_prev
        sigma = eta * np.sqrt((1.0 - ac_prev) / (1.0 - ac)) * np.sqrt(1.0 - ac / ac_prev)
        c = np.zeros((self.num_timesteps, 8), dtype=np.float32)
        c[:, 0] = self.sqrt_recip_alphas_cumprod
        c[:, 1] = self.sqrt_recipm1_alphas_cumprod
        c[:, 2] = np.sqrt(ac_prev)
        c[:, 3] = np.sqrt(np.maximum(0.0, 1.0 - ac_prev - sigma ** 2))
        c[:, 4] = sigma * (np.arange(self.num_timesteps) != 0)
        return c

    def inpaint_coef_table(self) -> np.ndarray:
        """[T+1, 2] fp32 rows consumed by cb2_plan_set_inpaint, computed in float64 and rounded once.  Row s < T is
        {sqrt(acp_prev[s]), sqrt(1 - acp_prev[s])}, the level a kept row takes after step s; row T is {sqrt(acp[T-1]),
        sqrt(1 - acp[T-1])}, its level before the first step.  Row 0 is exactly (1, 0), so kept rows end at their latent.
        The same table serves DDPM and DDIM on this respacing."""
        level = np.append(self.alphas_cumprod_prev, self.alphas_cumprod[-1])
        return np.stack([np.sqrt(level), np.sqrt(1.0 - level)], axis=1).astype(np.float32)

    def _coef_on(self, device, eta=None):
        """coef_table (eta None) or ddim_coef_table(eta) on `device`, uploaded once."""
        key = str(device) if eta is None else ("ddim", float(eta), str(device))
        if key not in self._coef_dev:
            table = self.coef_table() if eta is None else self.ddim_coef_table(eta)
            self._coef_dev[key] = torch.from_numpy(table).to(device)
        return self._coef_dev[key]

    # -- sampling ----------------------------------------------------------------------------------
    def p_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                      model_kwargs=None, device=None, progress=False, step_noise=None):
        """gaussian_diffusion.py:451-495.  `step_noise` [T, *shape] (extension) injects the per-step
        N(0,1) draws the reference takes from randn_like (:440); default: one torch.randn call."""
        from .latent_model import fused_sampler_for
        fused = fused_sampler_for(model)
        if fused is not None and cond_fn is None and denoised_fn is None and not clip_denoised:
            return fused.sample_loop(self, shape, noise, model_kwargs or {}, device, step_noise)
        final = None
        for final in self.p_sample_loop_progressive(model, shape, noise, clip_denoised, denoised_fn, cond_fn, model_kwargs,
                                                    device, progress, step_noise):
            pass
        return final["sample"]

    def p_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                                  model_kwargs=None, device=None, progress=False, step_noise=None):
        """gaussian_diffusion.py:497-547 (generic callable model; update on the GPU via cb2_p_sample)."""
        if cond_fn is not None or denoised_fn is not None or clip_denoised:
            raise NotImplementedError("cond_fn / denoised_fn / clip_denoised are not used by the reference's sampling path")
        N.require_cuda()
        device = torch.device(device if device is not None else "cuda")
        img = noise if noise is not None else torch.randn(*shape, device=device)
        img = img.to(device, torch.float32).contiguous()
        for i in list(range(self.num_timesteps))[::-1]:
            t = torch.tensor([i] * shape[0], device=device)
            n = step_noise[i].to(device, torch.float32).contiguous() if step_noise is not None else torch.randn_like(img)
            out = self.p_sample(model, img, t, clip_denoised=False, model_kwargs=model_kwargs, _noise=n)
            yield out
            img = out["sample"]

    def p_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None,
                 x_self_cond=None, _noise=None):
        """gaussian_diffusion.py:404-449: one reverse step; model(x, timestep_map[t], **kwargs) -> [B,...,2C]."""
        model_kwargs = model_kwargs or {}
        map_t = torch.tensor(self.timestep_map, device=t.device, dtype=t.dtype)[t]     # respace.py:124-125
        out = model(x, map_t, **model_kwargs).to(torch.float32).contiguous()
        C_ = x.shape[-1]
        rows = x.numel() // C_
        noise = _noise if _noise is not None else torch.randn_like(x)
        nxt = torch.empty_like(x)
        N.check(N.lib().cb2_p_sample(N.dptr(x.contiguous(), torch.float32), N.dptr(out), N.dptr(noise.contiguous(), torch.float32),
                                     N.dptr(self._coef_on(x.device)), N.dptr(t.to(torch.int32).contiguous()),
                                     rows // x.shape[0], rows, C_, N.dptr(nxt), N.stream_ptr()), "p_sample")
        eps = out[..., :C_]
        c = self._coef_on(x.device)[t].view(-1, *([1] * (x.dim() - 1)), 8)
        return {"sample": nxt, "pred_xstart": c[..., 2] * x - c[..., 3] * eps}

    # -- DDIM (IDDPM / DiT gaussian_diffusion.py ddim_sample*; the reference has no DDIM sampler) ---------------------
    @staticmethod
    def _check_ddim_args(clip_denoised, denoised_fn, cond_fn):
        if cond_fn is not None or denoised_fn is not None or clip_denoised:
            raise NotImplementedError("DDIM sampling supports clip_denoised=False without cond_fn / denoised_fn")

    def ddim_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None,
                         device=None, progress=False, eta=0.0, step_noise=None):
        """IDDPM ddim_sample_loop.  With eta = 0 the loop is deterministic and draws no per-step noise; otherwise
        `step_noise` [T, *shape] (extension, as in p_sample_loop) injects the N(0,1) draws, default one torch.randn call.
        A codlad_b200 denoiser runs the whole loop as one CUDA graph with the update fused into its last kernel."""
        self._check_ddim_args(clip_denoised, denoised_fn, cond_fn)
        from .latent_model import fused_sampler_for
        fused = fused_sampler_for(model)
        if fused is not None:
            return fused.sample_loop(self, shape, noise, model_kwargs or {}, device, step_noise, update="ddim", eta=eta)
        final = None
        for final in self.ddim_sample_loop_progressive(model, shape, noise, clip_denoised, denoised_fn, cond_fn, model_kwargs,
                                                       device, progress, eta, step_noise):
            pass
        return final["sample"]

    def ddim_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                                     model_kwargs=None, device=None, progress=False, eta=0.0, step_noise=None):
        """IDDPM ddim_sample_loop_progressive (generic callable model; update on the GPU via cb2_ddim_sample)."""
        self._check_ddim_args(clip_denoised, denoised_fn, cond_fn)
        N.require_cuda()
        device = torch.device(device if device is not None else "cuda")
        img = noise if noise is not None else torch.randn(*shape, device=device)
        img = img.to(device, torch.float32).contiguous()
        for i in list(range(self.num_timesteps))[::-1]:
            t = torch.tensor([i] * shape[0], device=device)
            n = None
            if eta != 0:
                n = step_noise[i].to(device, torch.float32).contiguous() if step_noise is not None else torch.randn_like(img)
            out = self.ddim_sample(model, img, t, clip_denoised=False, model_kwargs=model_kwargs, eta=eta, _noise=n)
            yield out
            img = out["sample"]

    def ddim_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None, eta=0.0, _noise=None):
        """IDDPM ddim_sample: one DDIM step; model(x, timestep_map[t], **kwargs) -> [B,...,2C] (the variance half is unused).
        Returns dict(sample, pred_xstart).  With eta = 0 no noise is drawn or read."""
        self._check_ddim_args(clip_denoised, denoised_fn, cond_fn)
        model_kwargs = model_kwargs or {}
        map_t = torch.tensor(self.timestep_map, device=t.device, dtype=t.dtype)[t]     # respace.py:124-125
        out = model(x, map_t, **model_kwargs).to(torch.float32).contiguous()
        C_ = x.shape[-1]
        rows = x.numel() // C_
        noise = None
        if eta != 0:
            noise = (_noise if _noise is not None else torch.randn_like(x)).contiguous()
        coef = self._coef_on(x.device, eta)
        nxt = torch.empty_like(x)
        N.check(N.lib().cb2_ddim_sample(N.dptr(x.contiguous(), torch.float32), N.dptr(out), N.dptr(noise, torch.float32), N.dptr(coef),
                                        N.dptr(t.to(torch.int32).contiguous()), rows // x.shape[0], rows, C_, N.dptr(nxt), N.stream_ptr()),
                "ddim_sample")
        c = coef[t].view(-1, *([1] * (x.dim() - 1)), 8)
        return {"sample": nxt, "pred_xstart": c[..., 0] * x - c[..., 1] * out[..., :C_]}

    def p_mean_variance(self, model, x, t, clip_denoised=True, denoised_fn=None, model_kwargs=None, x_self_cond=None):
        """gaussian_diffusion.py:262-360 for the shipped configuration (epsilon prediction, learned-range variance):
        dict(mean, variance, log_variance, pred_xstart).  Caller-facing glue for code that inspects one reverse step; the
        sampling loop itself never materialises these (they are fused into the final node kernel / cb2_p_sample)."""
        if denoised_fn is not None or clip_denoised:
            raise NotImplementedError("denoised_fn / clip_denoised are not used by the reference's sampling path")
        model_kwargs = model_kwargs or {}
        map_t = torch.tensor(self.timestep_map, device=t.device, dtype=t.dtype)[t]     # respace.py:124-125
        out = model(x, map_t, **model_kwargs).to(torch.float32)
        C_ = x.shape[-1]
        eps, v = out[..., :C_], out[..., C_:]
        c = self._coef_on(x.device)[t].view(-1, *([1] * (x.dim() - 1)), 8)
        frac = (v + 1) / 2
        log_variance = frac * c[..., 1] + (1 - frac) * c[..., 0]
        pred_xstart = c[..., 2] * x - c[..., 3] * eps
        mean = c[..., 4] * pred_xstart + c[..., 5] * x
        return {"mean": mean, "variance": torch.exp(log_variance), "log_variance": log_variance, "pred_xstart": pred_xstart}

    # -- loss values (evaluation only: the CUDA denoiser has no backward, so there is no training step here) ---------
    def _table_on(self, name, t, ndim):
        key = (name, str(t.device))
        if key not in self._coef_dev:
            self._coef_dev[key] = torch.from_numpy(getattr(self, name)).to(t.device).float()     # .float() as gaussian_diffusion.py:737
        return self._coef_dev[key][t].view(-1, *([1] * (ndim - 1)))

    def q_sample(self, x_start, t, noise=None):
        """gaussian_diffusion.py:223-238: x_t ~ q(x_t | x_0)."""
        noise = torch.randn_like(x_start) if noise is None else noise
        return (self._table_on("sqrt_alphas_cumprod", t, x_start.dim()) * x_start
                + self._table_on("sqrt_one_minus_alphas_cumprod", t, x_start.dim()) * noise)

    def q_posterior_mean_variance(self, x_start, x_t, t):
        """gaussian_diffusion.py:240-260: mean, variance and clipped log-variance of q(x_{t-1} | x_t, x_0)."""
        d = x_t.dim()
        mean = self._table_on("posterior_mean_coef1", t, d) * x_start + self._table_on("posterior_mean_coef2", t, d) * x_t
        shape = x_t.shape
        return (mean, self._table_on("posterior_variance", t, d).expand(shape),
                self._table_on("posterior_log_variance_clipped", t, d).expand(shape))

    @staticmethod
    def _mean_flat(x, mask=None):
        dims = list(range(1, x.dim()))
        return x.mean(dim=dims) if mask is None else (x * mask).sum(dim=dims) / mask.sum(dim=dims)      # gaussian_diffusion.py:16-26

    def _vb_terms_bpd(self, model, x_start, x_t, t, mask=None):
        """gaussian_diffusion.py:549-596: KL(q(x_{t-1}|x_t,x_0) || p(x_{t-1}|x_t)) in bits, the discretised decoder NLL at t = 0."""
        true_mean, _, true_logvar = self.q_posterior_mean_variance(x_start, x_t, t)
        out = self.p_mean_variance(model, x_t, t, clip_denoised=False)
        lv = out["log_variance"]
        kl = 0.5 * (-1.0 + lv - true_logvar + torch.exp(true_logvar - lv) + (true_mean - out["mean"]) ** 2 * torch.exp(-lv))   # diffusion_utils.py:10-37
        m = None if mask is None else mask.unsqueeze(-1).expand_as(x_start)
        kl = self._mean_flat(kl, m) / math.log(2.0)
        # discretised Gaussian log-likelihood, diffusion_utils.py:62-88 (tanh approximation of the normal CDF, bin half-width 1/255)
        cdf = lambda v: 0.5 * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (v + 0.044715 * torch.pow(v, 3))))
        centered, inv_std = x_start - out["mean"], torch.exp(-0.5 * lv)
        cdf_plus, cdf_min = cdf(inv_std * (centered + 1.0 / 255.0)), cdf(inv_std * (centered - 1.0 / 255.0))
        log_probs = torch.where(x_start < -0.999, torch.log(cdf_plus.clamp(min=1e-12)),
                                torch.where(x_start > 0.999, torch.log((1.0 - cdf_min).clamp(min=1e-12)),
                                            torch.log((cdf_plus - cdf_min).clamp(min=1e-12))))
        nll = self._mean_flat(-log_probs, m) / math.log(2.0)
        return {"output": torch.where(t == 0, nll, kl), "pred_xstart": out["pred_xstart"]}

    def training_losses(self, model, x_start, t, model_kwargs=None, noise=None):
        """gaussian_diffusion.py:598-725 for the shipped configuration (epsilon prediction, learned-range variance, MSE loss +
        VB term on the frozen mean): dict(mse, vb, loss), each [B].  Values only -- use it to score a checkpoint; `train_latent`
        itself (SURVEY.md section 8, row f-1) needs the backward pass of the denoiser, which this package does not have."""
        model_kwargs = dict(model_kwargs or {})
        model_kwargs.pop("epoch", None)
        noise = torch.randn_like(x_start) if noise is None else noise
        x_t = self.q_sample(x_start, t, noise)
        map_t = torch.tensor(self.timestep_map, device=t.device, dtype=t.dtype)[t]     # respace.py:124-125
        out = model(x_t, map_t, **model_kwargs).to(torch.float32)
        C_ = x_t.shape[-1]
        if out.shape != (*x_t.shape[:-1], 2 * C_):
            raise ValueError(f"model output {tuple(out.shape)}, expected {(*x_t.shape[:-1], 2 * C_)}")
        mask = model_kwargs.get("mask")
        vb = self._vb_terms_bpd(lambda *a, **k: out, x_start, x_t, t, mask)["output"]
        if self.loss_type == "rescaled_mse":
            vb = vb * (self.num_timesteps / 1000.0)
        diff2 = (noise - out[..., :C_]) ** 2
        mse = self._mean_flat(diff2, None if mask is None else mask.unsqueeze(-1).expand_as(diff2))
        return {"mse": mse, "vb": vb, "loss": mse + vb}


def create_diffusion(timestep_respacing, noise_schedule="linear", use_kl=False, rescale_learned_sigmas=False,
                     sigma_small=False, predict_xstart=False, learn_sigma=True, diffusion_steps=1000, self_condition=False):
    """diffusion_and_flow/__init__.py:10-60."""
    if timestep_respacing is None or timestep_respacing == "":
        timestep_respacing = [diffusion_steps]
    betas = get_named_beta_schedule(noise_schedule, diffusion_steps)
    if use_kl:
        raise NotImplementedError("the KL loss type is not used by the reference's training script")
    return SpacedDiffusion(space_timesteps(diffusion_steps, timestep_respacing), betas, learn_sigma=learn_sigma,
                           predict_xstart=predict_xstart, sigma_small=sigma_small, self_condition=self_condition,
                           loss_type="rescaled_mse" if rescale_learned_sigmas else "mse")
