"""`mpnn_diffusion` denoiser behind the reference's own call surface
(reference models/latent_model.py:78-281): same factory, same `state_dict()` keys and shapes
(108 tensors, so `torch.load(ckpt)["net_model" | "ema_model"]` loads, test.py:271-286), same
`forward(x, t, y, mask, batch, x_self_cond)` contract -- but the forward is the CUDA path of
libcodlad_b200.so.  There is no PyTorch implementation of the network in this package: without
the library / a CUDA device the module raises.

What the module does on the host is format conversion only: the reference batch dict
(`CG_nxyz [sum L, 4]`, `num_CGs [B]`, utils/dataset_module.py:259-295) becomes padded frames,
and the per-geometry plan (k-NN graph, edge features, h_E0 -- all functions of the C-alpha trace
alone) is cached across the 100 calls of a sampling loop instead of being recomputed per step
as the reference does (latent_model.py:208).
"""
from __future__ import annotations

import torch
from torch import nn

from . import batching, weights
from .engine import DenoiserEngine, Plan


class _Node(nn.Module):
    """Container used to give parameters the reference's dotted names."""


def _register(root: nn.Module, dotted: str, value: torch.Tensor):
    *path, leaf = dotted.split(".")
    mod = root
    for part in path:
        if part not in mod._modules:
            mod.add_module(part, _Node())
        mod = mod._modules[part]
    mod.register_parameter(leaf, nn.Parameter(value, requires_grad=False))


class ProteinMPNN_diffusion_new(nn.Module):
    """Drop-in for the reference class of the same name (latent_model.py:78-268), eval/sampling only."""

    def __init__(self, input_size: int = 3, hidden_dim: int = 128, k_neighbors: int = 64, unconditional: bool = True,
                 diffusion: str = "diffusion", self_condition: bool = False, class_dropout_prob: float = 0.1,
                 precision: str = "f16", init_seed: int = 0, **_ignored):
        super().__init__()
        if hidden_dim != 128 or input_size != 3:
            raise NotImplementedError("codlad_b200 implements the shipped configuration: hidden_dim=128, input_size=3")
        if self_condition:
            raise NotImplementedError("self-conditioning is not used by the reference's sampling path")
        self.input_size, self.k_neighbors, self.precision = input_size, int(k_neighbors), precision
        self.learn_sigma = diffusion == "diffusion"
        for name, t in weights.init_denoiser_state(init_seed, input_size=input_size).items():
            _register(self, name, t)
        self._engine = None
        self._plans = {}
        self._last = None
        self.eval()

    # -- packed device copy of the weights (rebuilt after load_state_dict) ---------------------------
    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        state_dict = {k.removeprefix("module."): v for k, v in state_dict.items()}     # test.py:277-285 retry
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self.refresh()
        return out

    def refresh(self):
        """Drop the packed weights and every cached plan (call after mutating parameters in place)."""
        for ent in self._plans.values():
            ent["plan"].close()
        self._plans.clear()
        self._last = None
        if self._engine is not None:
            self._engine.close()
        self._engine = None

    def engine(self) -> DenoiserEngine:
        if self._engine is None:
            self._engine = DenoiserEngine(self.state_dict(), self.k_neighbors)
        return self._engine

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("this module is the inference surface; the train_latent step (forward + backward + AdamW/EMA, SURVEY.md "
                                      "section 8 row f-1) is codlad_b200.train.DenoiserTrainer, which takes this module's state_dict()")
        return super().train(False)

    # -- geometry ------------------------------------------------------------------------------------
    def plan_for(self, batch: dict, n_members: int) -> Plan:
        """Plan for the frames of `batch` with `n_members` batch rows (n_members == F, or 2F for test.py's doubled
        batch, latent_model.py:178-186 / test.py:505-521).

        Plans are cached per GEOMETRY (F, n_members, Lmax) and remember the CONTENT they were built for: a new batch of
        the same shape (the next frames of the reference driver loop, test.py:481-534) re-runs the per-frame precompute
        on the existing plan instead of allocating a new one, and a batch is only taken as "the same" if it is the very
        tensor object the plan was built from (a held reference, so its storage cannot be recycled) at the same version,
        or if its bytes compare equal -- never by address alone."""
        cg, num = batch["CG_nxyz"], batch["num_CGs"]
        ent = self._last
        if (ent is not None and ent["cg_ref"] is cg and ent["num_ref"] is num and ent["version"] == (cg._version, num._version)
                and ent["n_members"] == int(n_members)):
            return ent["plan"]
        num_l = tuple(int(v) for v in num.tolist())
        F, L = len(num_l), max(num_l)
        if n_members % F != 0:
            raise ValueError(f"batch of {n_members} rows over {F} frames")
        cg_host = cg.detach().to("cpu", torch.float32)
        # frames of the batch that are byte-identical (an ensemble written as repeated frames, test.py's doubled batch) share one
        # k-NN graph / feature set: the plan holds the DISTINCT frames and maps every batch row to one of them
        X, z = batching.pad_frames(cg_host, torch.tensor(num_l), L)
        first, uniq, of_frame = {}, [], []
        for f in range(F):
            key = (num_l[f], X[f].numpy().tobytes(), z[f].numpy().tobytes())
            if key not in first:
                first[key] = len(uniq)
                uniq.append(f)
            of_frame.append(first[key])
        Fu = len(uniq)
        geo = (Fu, int(n_members), L)
        ent = self._plans.get(geo)
        if ent is None:
            if len(self._plans) >= 4:                  # a sampling run alternates between very few geometries
                self._plans.pop(next(iter(self._plans)))["plan"].close()
            ent = {"plan": Plan(self.engine(), Fu, int(n_members), L, self.precision), "cg": None, "num": None, "n_members": int(n_members),
                   "bufs": None, "schedule": None}
            self._plans[geo] = ent
        if ent["num"] != num_l or ent["cg"] is None or not torch.equal(ent["cg"], cg_host):
            frame_of = torch.tensor(of_frame, dtype=torch.int32).repeat(n_members // F)
            ent["plan"].set_frames(X[uniq].contiguous(), torch.tensor([num_l[f] for f in uniq], dtype=torch.int32), z[uniq].contiguous(), frame_of)
            ent["cg"], ent["num"] = cg_host.clone(), num_l
        ent["cg_ref"], ent["num_ref"], ent["version"] = cg, num, (cg._version, num._version)
        self._last = ent
        return ent["plan"]

    def _entry_of(self, plan: Plan) -> dict:
        for ent in self._plans.values():
            if ent["plan"] is plan:
                return ent
        raise KeyError("plan is not cached by this module")

    def forward(self, x, t, y=None, mask=None, batch=None, x_self_cond=None):
        """x [B, L, 3], t [B] (original 0..999 scale; int or float), mask [B, L] bool, batch = reference batch dict.
        `y` and `x_self_cond` are accepted and ignored exactly like the reference (SURVEY.md 8a, row a6).
        Returns [B, L, 6] (eps | variance logits); padded positions are unspecified."""
        if batch is None:
            raise ValueError("forward() needs the reference batch dict (CG_nxyz, num_CGs)")
        plan = self.plan_for(batch, x.shape[0])
        if x.shape[1] != plan.L:
            raise ValueError(f"x has L={x.shape[1]}, the batch has Lmax={plan.L}")
        return plan.forward(x, t.to(torch.float32))


class _FusedSampler:
    """Whole reverse-diffusion loop on the device (one CUDA graph) for a codlad_b200 denoiser."""

    def __init__(self, model: ProteinMPNN_diffusion_new):
        self.model = model

    def sample_loop(self, diffusion, shape, noise, model_kwargs, device, step_noise, update="ddpm", eta=0.0):
        """update "ddpm" (p_sample_loop) or "ddim" with `eta` (ddim_sample_loop; eta = 0 draws no step noise)."""
        batch = model_kwargs.get("batch")
        model = self.model
        plan = model.plan_for(batch, shape[0])
        ent = model._entry_of(plan)
        T = diffusion.num_timesteps
        ddim = update == "ddim"
        sched_key = (update, float(eta) if ddim else None, T, tuple(int(v) for v in diffusion.timestep_map))
        if ent["schedule"] != sched_key:                 # (re-)tabulate the adaLN rows only when the schedule changes: it drops the graph
            if ddim:
                plan.set_ddim_schedule(diffusion.timestep_map, diffusion.ddim_coef_table(eta))
            else:
                plan.set_schedule(diffusion.timestep_map, diffusion.coef_table())
            ent["schedule"] = sched_key
        noisy = not ddim or eta != 0
        dev = plan.device
        bufs = ent["bufs"]
        if bufs is None or (noisy and (bufs[1] is None or bufs[1].shape[0] != T)):
            # persistent x / noise buffers: the CUDA graph of the loop is keyed on them
            x = bufs[0] if bufs is not None else torch.empty(*shape, device=dev, dtype=torch.float32)
            bufs = ent["bufs"] = (x, torch.empty(T, *shape, device=dev, dtype=torch.float32) if noisy else None)
        x, eps = bufs[0], bufs[1] if noisy else None
        if noise is not None:
            x.copy_(noise, non_blocking=True)
        else:
            torch.randn(*shape, device=dev, out=x)
        if eps is not None:
            if step_noise is not None:
                eps.copy_(step_noise, non_blocking=True)
            else:
                torch.randn(T, *shape, device=dev, out=eps)
        plan.sample(x, eps, use_graph=True)
        return x.clone()                                 # the caller owns its result; the buffer is reused by the next call


def fused_sampler_for(model):
    """`model` as handed to p_sample_loop: the module itself or its bound `.forward` (test.py:533)."""
    owner = getattr(model, "__self__", model)
    return _FusedSampler(owner) if isinstance(owner, ProteinMPNN_diffusion_new) else None


def mpnn_diffusion(**kwargs):
    """latent_model.py:276-281: the factory fixes augment_eps=0, decoder_mask=False, use_seq_in_encoder=True."""
    return ProteinMPNN_diffusion_new(**kwargs)


MPNN_models = {"mpnn_diffusion": mpnn_diffusion}
