"""Ensemble-batched sampling driver: the B200 replacement of test.py's loop 2-4
(reference test.py:455-582; SURVEY.md section 8 row f-2).

Differences from the reference driver, none of which change results:
  * ensemble members are folded into the batch (the reference runs them sequentially);
  * no `cat([z, z])` batch doubling (test.py:505,533 computes every sample twice and discards half);
  * the k-NN graph / edge features / h_E0 are computed once per frame, the adaLN table once per
    schedule, and the 100-step loop is one CUDA graph;
  * the decode side (de-normalise, VQ, IC decoder, ic_to_xyz) runs on the same plan.

Host work here is input-format conversion only (padding, CSR of the given CG_nbr_list, slot maps).
"""
from __future__ import annotations

import math
import numbers
from dataclasses import dataclass, field

import torch

from . import batching, distributed, metrics, topology, weights
from .diffusion import create_diffusion
from .engine import (DenoiserEngine, Plan, VaeEngine, check_clash_args, check_keyed_normal_args, check_relax_args, check_start_steps,
                     keyed_normal)

VAE_DATA = {"N6": "PED", "K3": "PDB", "K4": "Atlas"}


def clash_pair_totals(counts: torch.Tensor) -> torch.Tensor:
    """Clashing atom pairs per member (int64 [NB]) from per-residue counts [NB, L], where every pair counts for both residues."""
    return counts.sum(1, dtype=torch.int64) // 2


def repair_accept(prev_pairs: torch.Tensor, new_pairs: torch.Tensor) -> torch.Tensor:
    """The acceptance rule of Backmapper.repair, per member: take the resampled latent only if it has fewer clashing pairs."""
    return new_pairs < prev_pairs


def trajectory_chunks(n_frames: int, chunks: int):
    """Split n_frames consecutive frames into `chunks` contiguous runs whose lengths differ by at most one, longer runs first.
    Returns [(first frame, length)]."""
    if isinstance(chunks, bool) or not isinstance(chunks, numbers.Integral) or chunks < 1:
        raise ValueError(f"chunks must be a positive integer, got {chunks!r}")
    if chunks > n_frames:
        raise ValueError(f"chunks ({chunks}) exceeds the number of frames ({n_frames})")
    q, r = divmod(int(n_frames), int(chunks))
    runs, start = [], 0
    for c in range(chunks):
        n = q + (1 if c < r else 0)
        runs.append((start, n))
        start += n
    return runs


def trajectory_args(T: int, n_frames: int, num_ensemble, steps, chunks):
    """Checks of the trajectory methods for a T-step schedule; returns (steps, runs) with the default steps = T // 4 and
    runs = trajectory_chunks(n_frames, chunks)."""
    if isinstance(num_ensemble, bool) or not isinstance(num_ensemble, numbers.Integral) or num_ensemble < 1:
        raise ValueError(f"num_ensemble must be a positive integer, got {num_ensemble!r}")
    steps = max(1, T // 4) if steps is None else steps
    check_start_steps(steps)
    if not 1 <= steps <= T:
        raise ValueError(f"steps must be in [1, {T}], got {steps}")
    return steps, trajectory_chunks(n_frames, chunks)


RELAX_ITERATIONS = 50       # default iterations of Backmapper.relax: planted 0.4 A overlaps are pushed past the threshold in them


def relax_option(relax):
    """The `relax=` option of the trajectory methods: None (no relaxation) or a dict with the keys `iterations` and `threshold` of
    Backmapper.relax, both optional.  Returns the full keyword dict (or None); raises ValueError; touches no device."""
    if relax is None:
        return None
    if not isinstance(relax, dict) or not set(relax) <= {"iterations", "threshold"}:
        raise ValueError(f"relax must be None or a dict with the keys 'iterations' and 'threshold', got {relax!r}")
    opts = {"iterations": RELAX_ITERATIONS, "threshold": 1.2, **relax}
    check_relax_args(opts["threshold"], opts["iterations"])
    return opts


def check_coords_args(ca_full, restype):
    """The input checks of Backmapper.backmap_coords: ca_full float32 [n_frames, L+2, 3] (n_frames, L >= 1) on the host or the
    current CUDA device, restype integer [L+2]."""
    if not torch.is_tensor(ca_full) or ca_full.dtype != torch.float32 or ca_full.dim() != 3 or ca_full.shape[2] != 3 \
            or ca_full.shape[0] < 1 or ca_full.shape[1] < 3:
        raise ValueError("ca_full must be a float32 tensor of shape [n_frames, L+2, 3] with n_frames >= 1 and L >= 1")
    if ca_full.device.type not in ("cpu", "cuda") or (ca_full.is_cuda and ca_full.device.index not in (None, torch.cuda.current_device())):
        raise ValueError("ca_full must be a host tensor or on the current CUDA device")
    L = ca_full.shape[1] - 2
    if not torch.is_tensor(restype) or restype.dtype.is_floating_point or restype.dtype.is_complex or restype.dtype == torch.bool \
            or tuple(restype.shape) != (L + 2,):
        raise ValueError(f"restype must be an integer tensor of shape {(L + 2,)}")


def residue_atom_ranges(fs: "FrameSet"):
    """The atoms of every real residue of every member of `fs`, gathered through slot_atom into contiguous ranges.  Returns
    (atoms int64 [A], counts int64 [R], rows int64 [R]): residue r = row rows[r] of the flattened [NB, L] grid owns
    atoms[sum(counts[:r]) : sum(counts[:r + 1])], rows of the output xyz laid out as decode writes it, in slot order.  Padded rows
    and residues without atoms are left out, so no range is empty."""
    fo = fs.frame_of.long().cpu()
    slots = fs.slot_atom.cpu().view(fs.F, fs.L, topology.SLOTS_PER_RESIDUE)[fo]                  # [NB, L, 14]
    valid = torch.arange(fs.L)[None] < fs.lengths.cpu().long()[fo][:, None]                      # [NB, L]
    present = (slots >= 0) & valid[..., None]
    counts = present.sum(-1).flatten()
    rows = torch.nonzero(counts > 0).squeeze(1)
    atoms = (slots.long() + fs.out_off.cpu().long()[:, None, None])[present]      # row-major: each residue's atoms in one run
    return atoms, counts[rows], rows


MEMBER_BITS = 16            # member key = frame key * 2^16 + ensemble index
FRAME_KEY_LIMIT = 1 << 47   # frame keys in [0, 2^47) keep every member key a non-negative int64


def member_keys(fs: "FrameSet", frame_keys=None) -> torch.Tensor:
    """Keys of the keyed sampling noise (engine.keyed_normal), host int64 [NB]: key_b = frame_keys[frame_of[b]] * 2^16 + e_b, where
    e_b counts the members of b's frame that come before b in member order.  frame_keys [F] defaults to arange(F); a caller that
    samples part of a larger job passes the frames' indices in that job, so a member gets the same noise as there.  For
    frames_from_batch(..., num_ensemble), where b = e * F + f, key_b = f * 2^16 + e."""
    fo = fs.frame_of.detach().cpu().long()
    if frame_keys is None:
        frame_keys = torch.arange(fs.F, dtype=torch.int64)
    else:
        frame_keys = torch.as_tensor(frame_keys).detach().cpu()
        if frame_keys.dtype.is_floating_point or frame_keys.dtype.is_complex or frame_keys.dtype == torch.bool \
                or tuple(frame_keys.shape) != (fs.F,):
            raise ValueError(f"frame_keys must be an integer sequence of length {fs.F}")
        frame_keys = frame_keys.long()
    order = torch.sort(fo, stable=True).indices                         # members grouped by frame, member order kept within a frame
    counts = torch.bincount(fo, minlength=fs.F)
    ens = torch.empty_like(fo)
    ens[order] = torch.arange(fs.NB) - (torch.cumsum(counts, 0) - counts)[fo[order]]
    return _compose_keys(frame_keys[fo], ens)


def unit_keys(units) -> torch.Tensor:
    """member_keys for a list of (frame, ensemble index) units of a job: host int64 [len(units)], key = frame * 2^16 + e, the key
    the unit gets from member_keys in a single frames_from_batch of the whole job (b = e * F + f).  ShardedBackmapper keys each
    rank's units with it."""
    t = torch.tensor([[int(f), int(e)] for f, e in units], dtype=torch.int64).view(-1, 2)
    if bool((t[:, 0] < 0).any()) or bool((t[:, 1] < 0).any()):
        raise ValueError("frame and ensemble indices of the units must be non-negative")
    return _compose_keys(t[:, 0], t[:, 1])


def _compose_keys(frame_keys: torch.Tensor, ens: torch.Tensor) -> torch.Tensor:
    """frame_keys * 2^16 + ens (int64), refusing what would make two members share a key: a frame key outside [0, 2^47) or an
    ensemble index of 2^16 or more."""
    if bool(((frame_keys < 0) | (frame_keys >= FRAME_KEY_LIMIT)).any()):
        raise ValueError("frame keys must lie in [0, 2^47)")
    if ens.numel() and int(ens.max()) >= 1 << MEMBER_BITS:
        raise ValueError(f"a frame holds {int(ens.max()) + 1} members; member keys allow at most 2^16 per frame")
    return frame_keys * (1 << MEMBER_BITS) + ens


@dataclass
class FrameSet:
    """Host-side description of F frames (equal padded length L) and the members sampled on them."""
    X: torch.Tensor            # [F, L, 3] trimmed C-alpha, zero padded
    ca_full: torch.Tensor      # [F, L+2, 3]
    cg_z: torch.Tensor         # [F, L] int32 residue-type ids
    lengths: torch.Tensor      # [F] int32
    csr_row: torch.Tensor      # [F*L+1] int32
    csr_col: torch.Tensor      # [E] int32
    orders: torch.Tensor       # [F, L, 10, 3] int8
    slot_atom: torch.Tensor    # [F, L*14] int32
    num_atoms: torch.Tensor    # [F] int64
    frame_of: torch.Tensor     # [NB] int32
    out_off: torch.Tensor = field(default=None)   # [NB] int64
    total_atoms: int = 0

    def __post_init__(self):
        na = self.num_atoms[self.frame_of.long()]
        self.out_off = torch.cumsum(na, 0) - na
        self.total_atoms = int(na.sum())

    _HOST_FIELDS = ("X", "ca_full", "cg_z", "lengths", "csr_row", "csr_col", "orders", "slot_atom", "frame_of", "out_off")

    def pin(self):
        """Page-lock the host tensors so uploads are true async DMA (what bench.py's e2e leg times)."""
        for name in self._HOST_FIELDS:
            t = getattr(self, name).contiguous()
            setattr(self, name, t.pin_memory() if torch.cuda.is_available() and not t.is_pinned() else t)
        return self

    def host_bytes(self) -> int:
        """Bytes copied host -> device by Backmapper.upload()."""
        return sum(getattr(self, n).numel() * getattr(self, n).element_size() for n in self._HOST_FIELDS)

    @property
    def F(self): return self.X.shape[0]
    @property
    def L(self): return self.X.shape[1]
    @property
    def NB(self): return self.frame_of.numel()


def frames_from_batch(batch: dict, infos, num_ensemble: int = 1, frame_of=None) -> FrameSet:
    """Convert a reference-schema batch dict (CG_collate, utils/dataset_module.py:259-295) of F frames
    plus their `info` tuples (one per frame, or one shared) into a FrameSet with `num_ensemble`
    members per frame (member order: ensemble-major, i.e. b = e*F + f), or with the explicit member list
    `frame_of` [NB] (frame index of every member; frames may then carry different member counts)."""
    num = batch["num_CGs"].to(torch.int64).cpu()
    if num.numel() == 0:
        raise ValueError("frames_from_batch: the batch holds no frames")
    if int(num.min()) < 1:
        raise ValueError("frames_from_batch: a frame with no residues")
    if frame_of is None and int(num_ensemble) < 1:
        raise ValueError("frames_from_batch: num_ensemble must be at least 1")
    F, L = num.numel(), int(num.max())
    cg = batch["CG_nxyz"].cpu().to(torch.float32)
    og = batch["OG_CG_nxyz"].cpu().to(torch.float32)
    if cg.shape[0] != int(num.sum()) or og.shape[0] != int(num.sum()) + 2 * F:
        raise ValueError("frames_from_batch: CG_nxyz / OG_CG_nxyz do not match num_CGs")
    shared = isinstance(infos, tuple) and len(infos) == 3 and torch.is_tensor(infos[0])
    if not shared and len(infos) != F:
        raise ValueError(f"frames_from_batch: {len(infos)} topology tuples for {F} frames")
    X, cg_z = batching.pad_frames(cg, num, L)
    ca_full = batching.pad_frames(og, num + 2, L + 2)[0]
    orders, slot_atom, num_atoms = _topology_tables(infos, shared, num, L)
    csr_row, csr_col = batching.batch_csr(batch["CG_nbr_list"], num, L)
    if frame_of is None:
        frame_of = torch.arange(F, dtype=torch.int32).repeat(num_ensemble)
    frame_of = torch.as_tensor(frame_of, dtype=torch.int32)
    return FrameSet(X, ca_full, cg_z, num.to(torch.int32), csr_row, csr_col, orders, slot_atom, num_atoms, frame_of)


def _topology_tables(infos, shared: bool, num: torch.Tensor, L: int):
    """Decoder topology of F frames of lengths num [F] padded to L: (orders [F,L,10,3] int8, slot_atom [F,L*14] int32,
    num_atoms [F] int64), from one shared info tuple or one per frame."""
    F = num.numel()
    orders = torch.zeros(F, L, 10, 3, dtype=torch.int8)
    orders[..., 1], orders[..., 2] = 1, 2
    slot_atom = torch.full((F, L * 14), -1, dtype=torch.int32)
    num_atoms = torch.zeros(F, dtype=torch.int64)
    if shared and bool((num == num[0]).all()):
        n = int(num[0])
        orders[:, :n] = infos[2].permute(1, 0, 2).to(torch.int8)[None]
        slot_atom[:, :n * 14] = topology.slot_to_atom_map(infos, n)[None]
        num_atoms[:] = infos[0].numel()
    else:
        per_frame = [infos] * F if shared else infos
        for f in range(F):
            n = int(num[f])
            permute, _, atom_orders = per_frame[f]
            orders[f, :n] = atom_orders.permute(1, 0, 2).to(torch.int8)
            slot_atom[f, :n * 14] = topology.slot_to_atom_map(per_frame[f], n)
            num_atoms[f] = permute.numel()
    return orders, slot_atom, num_atoms


def frames_from_coords(ca_full: torch.Tensor, restype: torch.Tensor, info, num_ensemble: int = 1) -> FrameSet:
    """FrameSet of F frames of one protein given as coordinates: ca_full [F, L+2, 3] (the coordinate columns of OG_CG_nxyz per
    frame, termini included), restype [L+2] (its residue ids), info the shared topology tuple; `num_ensemble` members per frame as in
    frames_from_batch, which it equals on every field except the radius graph: csr_row is all zero and csr_col empty, because the
    graph is meant to be built on the device (Backmapper.update_coords).  Host tensors."""
    ca_full = ca_full.detach().cpu().to(torch.float32).contiguous()
    F, L = ca_full.shape[0], ca_full.shape[1] - 2
    num = torch.full((F,), L, dtype=torch.int64)
    cg_z = restype.detach().cpu()[1:-1].to(torch.int32)[None].expand(F, L).contiguous()
    orders, slot_atom, num_atoms = _topology_tables(info, True, num, L)
    frame_of = torch.arange(F, dtype=torch.int32).repeat(num_ensemble)
    return FrameSet(ca_full[:, 1:-1].contiguous(), ca_full, cg_z, num.to(torch.int32), torch.zeros(F * L + 1, dtype=torch.int32),
                    torch.zeros(0, dtype=torch.int32), orders, slot_atom, num_atoms, frame_of)


class Backmapper:
    """CG trace -> all-atom ensemble: 100-step latent diffusion + VQ-VAE decode + IC reconstruction.
    sampler="ddpm" is the reference's ancestral sampler; sampler="ddim" uses IDDPM's DDIM update with `eta` on the same
    respacing (eta = 0: deterministic, no per-step noise is drawn or stored)."""

    def __init__(self, denoiser_state: dict, vae_state: dict, vae_type: str = "N6", k_neighbors: int = 64,
                 num_sampling_steps: int = 100, precision: str = "f16", latent_stats=None, max_plans: int = 4,
                 sampler: str = "ddpm", eta: float = 0.0):
        if sampler not in ("ddpm", "ddim"):
            raise ValueError(f"sampler must be 'ddpm' or 'ddim', got {sampler!r}")
        if sampler == "ddpm" and eta != 0:
            raise ValueError("eta applies to sampler='ddim' only")
        self.sampler, self.eta = sampler, float(eta)
        self.precision = precision
        self.k_neighbors = int(k_neighbors)
        self.max_plans = int(max_plans)
        self.denoiser = DenoiserEngine(denoiser_state, k_neighbors)
        stats = latent_stats or weights.LATENT_STATS[(vae_type, VAE_DATA[vae_type])]
        self.vae = VaeEngine(vae_state, stats[0], stats[1], angle_variant=vae_type in ("K3", "K4"))
        self.diffusion = create_diffusion(str(num_sampling_steps))
        self.T = self.diffusion.num_timesteps
        self._plans = {}
        self._bufs = {}
        self._keys = {}                 # id(plan) -> (host keys, the same on the device) of the plan's last seeded pass
        self._host_xyz = {}

    def plan_for(self, fs: FrameSet, keep_debug: bool = False) -> Plan:
        key = (fs.F, fs.NB, fs.L, keep_debug)
        plan = self._plans.get(key)
        if plan is None:
            while len(self._plans) >= self.max_plans:              # a plan owns every buffer of its geometry: keep few of them
                old = self._plans.pop(next(iter(self._plans)))
                self._bufs.pop(id(old), None)
                self._keys.pop(id(old), None)
                old.close()
            plan = Plan(self.denoiser, fs.F, fs.NB, fs.L, self.precision, keep_debug)
            if self.sampler == "ddim":
                plan.set_ddim_schedule(self.diffusion.timestep_map, self.diffusion.ddim_coef_table(self.eta))
            else:
                plan.set_schedule(self.diffusion.timestep_map, self.diffusion.coef_table())
        else:
            self._plans.pop(key)                                   # re-insert: most recently used last
        self._plans[key] = plan
        return plan

    def upload(self, fs: FrameSet, keep_debug: bool = False) -> Plan:
        """Host -> device: coordinates, graph, topology; then the per-frame precompute (k-NN, h_E0, filters)."""
        plan = self.plan_for(fs, keep_debug)
        plan.set_frames(fs.X, fs.lengths, fs.cg_z, fs.frame_of)
        plan.set_topology(self.vae, fs.ca_full, fs.csr_row, fs.csr_col, fs.orders, fs.slot_atom, fs.out_off)
        return plan

    def sample(self, plan: Plan, fs: FrameSet, z: torch.Tensor = None, step_noise: torch.Tensor = None,
               use_graph: bool = True, generator: torch.Generator = None, seed: int = None, keys: torch.Tensor = None, draw: int = 0):
        """Device-resident path: returns dict(latent, idx, ic_recon, xyz) of CUDA tensors.
        z [NB,L,3] initial noise, step_noise [T,NB,L,3]; drawn on the device when omitted, from `generator` or, with `seed`, as
        keyed noise (engine.keyed_normal): member b gets slices 0 (z) and 1 + s (the noise of step s) of its key keys[b] (int64 [NB],
        default member_keys(fs)) and `draw`, the same in any batch that holds it.  seed excludes generator, z and step_noise.
        DDIM with eta = 0 uses no step noise: `step_noise` is ignored.  Every residue is sampled anew, also after resample() on
        the same plan."""
        self._check_noise_args(fs, z, step_noise, generator, seed, keys, draw)
        plan.clear_inpaint()
        plan.set_start(0)
        return self._sample(plan, fs, z, step_noise, use_graph, generator, None, seed, keys, draw)

    def resample(self, plan: Plan, fs: FrameSet, latent: torch.Tensor, keep: torch.Tensor, z: torch.Tensor = None,
                 step_noise: torch.Tensor = None, generator: torch.Generator = None, seed: int = None, keys: torch.Tensor = None,
                 draw: int = 0):
        """Latent inpainting: keep the residues of an earlier pass where keep [NB,L] (bool) is True and sample the others
        anew, conditioned on the kept ones through the denoiser.  latent [NB,L,3] is that pass's normalised latent
        (`sample(...)["latent"]`, which may be passed as is).  Kept rows follow the forward marginal of their latent with the
        fixed draw z and end at it exactly, so they keep their VQ index.  z, step_noise, generator, seed, keys and draw as in
        sample().  Returns the same dict as sample()."""
        self._check_noise_args(fs, z, step_noise, generator, seed, keys, draw)
        self._check_latent_keep(plan, fs, latent, keep)
        plan.set_inpaint(keep, latent, self.diffusion.inpaint_coef_table())      # copies latent before z overwrites its buffer
        plan.set_start(0)
        return self._sample(plan, fs, z, step_noise, True, generator, None, seed, keys, draw)

    def refine(self, plan: Plan, fs: FrameSet, latent: torch.Tensor, steps: int, keep: torch.Tensor = None, z: torch.Tensor = None,
               step_noise: torch.Tensor = None, generator: torch.Generator = None, seed: int = None, keys: torch.Tensor = None,
               draw: int = 0):
        """Partial-noise refinement (SDEdit): noise the normalised latent [NB,L,3] to the level of respaced step `steps` with the
        draw z, x = sqrt(acp[steps-1]) latent + sqrt(1 - acp[steps-1]) z, and run only the last `steps` of the T steps,
        conditioned on the frames of `fs` as uploaded now.  The strength is steps / T, with 1 <= steps <= T.  latent may be
        `sample(...)["latent"]` as it is.  keep [NB,L] (bool) keeps those residues exactly, as resample() does; None refines every
        residue.  z [NB,L,3] and step_noise [T,NB,L,3] (slices [0, steps) are read) are drawn when omitted; DDIM with eta = 0 uses
        no step noise.  With `seed` the keyed slices 0 and 1 .. steps are filled, the ones a full pass would use for z and those
        steps (generator, seed, keys and draw as in sample()).  Returns the same dict as sample(); a later sample() or resample()
        is a full pass again."""
        self._check_noise_args(fs, z, step_noise, generator, seed, keys, draw)
        check_start_steps(steps)
        if not 1 <= steps <= self.T:
            raise ValueError(f"steps must be in [1, {self.T}], got {steps}")
        if keep is None:
            keep = torch.zeros(fs.NB, fs.L, dtype=torch.bool, device=plan.device)
        self._check_latent_keep(plan, fs, latent, keep)
        plan.set_inpaint(keep, latent, self.diffusion.inpaint_coef_table())
        plan.set_start(steps)
        return self._sample(plan, fs, z, step_noise, True, generator, steps, seed, keys, draw)

    @staticmethod
    def _check_noise_args(fs: FrameSet, z, step_noise, generator, seed, keys, draw):
        """seed is one source of noise, generator / z / step_noise another; keys [NB] (int64) and draw belong to seed."""
        if seed is None:
            if keys is not None or draw != 0:
                raise ValueError("keys and draw select keyed noise: they need a seed")
            return
        if generator is not None or z is not None or step_noise is not None:
            raise ValueError("seed draws z and the step noise itself: it excludes generator, z and step_noise")
        check_keyed_normal_args(seed, fs.L, draw, 0, 1)
        if keys is not None and (not torch.is_tensor(keys) or keys.dtype != torch.int64 or tuple(keys.shape) != (fs.NB,)):
            raise ValueError(f"keys must be an int64 tensor of shape {(fs.NB,)}")

    @staticmethod
    def _check_latent_keep(plan: Plan, fs: FrameSet, latent, keep):
        shape = (fs.NB, fs.L, 3)
        if not torch.is_tensor(latent) or latent.dtype != torch.float32 or tuple(latent.shape) != shape:
            raise ValueError(f"latent must be a float32 tensor of shape {shape}")
        if not torch.is_tensor(keep) or keep.dtype != torch.bool or tuple(keep.shape) != shape[:2]:
            raise ValueError(f"keep must be a bool tensor of shape {shape[:2]}")
        if latent.device != plan.device or keep.device != plan.device:
            raise ValueError(f"latent and keep must be on {plan.device}")

    def residue_clashes(self, plan: Plan, fs: FrameSet, xyz: torch.Tensor, threshold: float = 1.2, grow: int = 0):
        """Per-residue clashes of a decoded sample, on the device (cb2_plan_residue_clashes): clash_result's criterion
        (test.py:118-139) per residue, with no reference structure.  xyz [fs.total_atoms, 3] as sample() returns it.  Returns
        (counts int32 [NB, L], keep bool [NB, L]): counts[b, i] = atom pairs of residue i with other residues of member b closer
        than `threshold` Angstrom, the peptide bond C(i)-N(i+1) left out (each pair counts for both residues); keep is False
        where residue i or one of its `grow` nearest other residues (the plan's k-NN graph) clashes -- the mask resample() takes."""
        shape = (fs.total_atoms, 3)
        if not torch.is_tensor(xyz) or xyz.dtype != torch.float32 or tuple(xyz.shape) != shape:
            raise ValueError(f"xyz must be a float32 tensor of shape {shape}")
        if xyz.device != plan.device:
            raise ValueError(f"xyz must be on {plan.device}")
        return plan.residue_clashes(xyz, threshold, grow)

    def repair(self, plan: Plan, fs: FrameSet, out: dict, max_rounds: int = 3, grow: int = 0, threshold: float = 1.2,
               generator: torch.Generator = None, seed: int = None, keys: torch.Tensor = None):
        """Clash-driven repair of a backmapped sample `out` (the dict of sample() / resample()): each round flags the clashing
        residues (residue_clashes), stops when no member has a clash, and otherwise resamples the flagged residues of every
        member with latent inpainting, fresh noise from `generator`, or with `seed` the keyed noise of draw r + 1 in round r
        (keys as in sample()), so a member's rounds draw what they would in any other batch.  Per member the new latent is accepted
        only when its number of clashing pairs went down; otherwise the member keeps its previous latent.  The accepted latents are
        decoded once at the end.  Kept residues keep their latent and VQ index; their coordinates can still move where the IC
        decoder's radius graph reaches a regenerated neighbour.  A round costs one resample pass (one sampling pass plus decode).
        Returns the dict of sample() plus `clashes` (int32 [NB, L], the counts of the returned structure) and `clash_pairs`
        (int64 [rounds run + 1, NB], clashing pairs per member; row 0 is the input's).  The plan is left for plain sample()."""
        if not isinstance(out, dict) or not all(k in out for k in ("latent", "idx", "zq", "ic_recon", "xyz")):
            raise ValueError("out must be the dict returned by sample() or resample()")
        if isinstance(max_rounds, bool) or not isinstance(max_rounds, int) or max_rounds < 0:
            raise ValueError(f"max_rounds must be a non-negative integer, got {max_rounds!r}")
        check_clash_args(threshold, grow, plan.K)
        self._check_noise_args(fs, None, None, generator, seed, keys, 0)
        shape = (fs.NB, fs.L, 3)
        latent = out["latent"]
        if not torch.is_tensor(latent) or latent.dtype != torch.float32 or tuple(latent.shape) != shape or latent.device != plan.device:
            raise ValueError(f"out['latent'] must be a float32 tensor of shape {shape} on {plan.device}")
        counts, keep = self.residue_clashes(plan, fs, out["xyz"], threshold, grow)
        pairs = clash_pair_totals(counts)
        rows = [pairs]
        latent = latent.clone()                  # resample() writes the plan's latent buffer, which out["latent"] may be
        for r in range(max_rounds):
            if not bool((pairs > 0).any()):
                break
            new = self.resample(plan, fs, latent, keep, generator=generator, seed=seed, keys=keys, draw=0 if seed is None else r + 1)
            new_counts, new_keep = self.residue_clashes(plan, fs, new["xyz"], threshold, grow)
            new_pairs = clash_pair_totals(new_counts)
            acc = repair_accept(pairs, new_pairs)
            latent = torch.where(acc[:, None, None], new["latent"], latent)
            keep = torch.where(acc[:, None], new_keep, keep)
            pairs = torch.where(acc, new_pairs, pairs)
            rows.append(pairs)
        plan.clear_inpaint()
        if len(rows) == 1:                       # nothing resampled: the input as it is
            res = dict(out)
        else:
            idx, zq, ic, xyz = plan.decode(self.vae, latent, denorm=True, num_atoms_total=fs.total_atoms)
            res = {"latent": latent, "idx": idx, "zq": zq, "ic_recon": ic, "xyz": xyz}
            counts, _ = self.residue_clashes(plan, fs, xyz, threshold, grow)
        res["clashes"] = counts
        res["clash_pairs"] = torch.stack(rows, 0)
        return res

    def relax(self, plan: Plan, fs: FrameSet, out: dict, iterations: int = RELAX_ITERATIONS, threshold: float = 1.2):
        """Restrained clash relaxation of a backmapped sample `out` (the dict of sample() / resample() / refine() / repair()), on the
        device (cb2_plan_relax): pushes atoms of different residues that are closer than `threshold` apart while holding the decoded
        bonded geometry and the C-alpha trace.  Per member: the C-alphas never move; every intra-residue pair within 3 A at the input
        (bonds, angles, ring closures) and the peptide pairs C(i)-N(i+1), CA(i)-N(i+1), O(i)-N(i+1), C(i)-CA(i+1) are restrained to
        their input distance d0; every other pair of two residues closer than c = threshold + 0.2 A is repelled.  It minimises
        E = sum 1.0 (d - d0)^2 + sum 10.0 (c - d)^2 with `iterations` capped steepest-descent steps (0.05 A^2 per unit force, at most
        0.1 A per atom and step), a fixed amount of work with no early exit.  Deterministic, and a member's result does not depend on
        its batch; a member with no pair closer than c comes back bit for bit.  Intra-residue overlaps are left as decoded.
        threshold must lie in (0, 2.0] A: above that the repulsion distance would reach the restrained 1-3 distances of the peptide
        (about 2.25-2.45 A).  0 <= iterations <= 10^5.
        Returns dict(out) with `xyz` replaced by the relaxed coordinates; `latent`, `idx` and `zq` are unchanged, so refine() and
        repair() can continue from them, and `ic_recon` still describes the unrelaxed decode.  Adds `clash_pairs` (int64 [2, NB]: pairs
        under `threshold` per member before and after, residue_clashes), `clashes` (int32 [NB, L], the counts after), `max_shift`
        (float32 [NB], the largest distance an atom moved) and `max_restraint_dev` (float32 [NB], the largest |d - d0|)."""
        if not isinstance(out, dict) or not all(k in out for k in ("latent", "idx", "zq", "ic_recon", "xyz")):
            raise ValueError("out must be the dict returned by sample(), resample(), refine() or repair()")
        check_relax_args(threshold, iterations)
        before, _ = self.residue_clashes(plan, fs, out["xyz"], threshold)
        xyz, shift, dev = plan.relax(out["xyz"], threshold, iterations)
        after, _ = self.residue_clashes(plan, fs, xyz, threshold)
        res = dict(out)
        res.update(xyz=xyz, clashes=after, clash_pairs=torch.stack((clash_pair_totals(before), clash_pair_totals(after)), 0),
                   max_shift=shift, max_restraint_dev=dev)
        return res

    def residue_motion(self, fs: FrameSet, xyz_a: torch.Tensor, xyz_b: torch.Tensor) -> torch.Tensor:
        """Per-residue RMSD between two decoded structures of the same frame set (xyz [fs.total_atoms, 3] CUDA float32, as
        sample() returns them), each residue's atoms superposed on their own (cb2_superposed_rmsd over the residue_atom_ranges).
        Returns float64 [NB, L] on the device, NaN on padded rows.  Between consecutive frames of a trajectory it measures
        side-chain flicker; between a sample and its refine() or repair() it shows what the pass changed."""
        shape = (fs.total_atoms, 3)
        for name, t in (("xyz_a", xyz_a), ("xyz_b", xyz_b)):
            if not torch.is_tensor(t) or t.dtype != torch.float32 or tuple(t.shape) != shape or not t.is_cuda:
                raise ValueError(f"{name} must be a CUDA float32 tensor of shape {shape}")
        if xyz_a.device != xyz_b.device:
            raise ValueError("xyz_a and xyz_b must be on the same device")
        atoms, counts, rows = residue_atom_ranges(fs)
        out = torch.full((fs.NB * fs.L,), math.nan, dtype=torch.float64, device=xyz_a.device)
        if rows.numel():
            atoms = atoms.to(xyz_a.device)
            out[rows.to(xyz_a.device)] = metrics.superposed_rmsd(xyz_a[atoms], xyz_b[atoms], counts)
        return out.view(fs.NB, fs.L)

    def backmap_trajectory(self, batches, info, num_ensemble: int = 1, steps: int = None, chunks: int = 1,
                           generator: torch.Generator = None, seed: int = None, relax: dict = None) -> torch.Tensor:
        """Backmap consecutive frames of one protein with warm starts.  batches: one reference-schema batch dict per frame (one
        frame each, all of the same length), info: the shared topology tuple.  The frames are split into `chunks` contiguous runs
        (trajectory_chunks) that go through one plan together, each run with `num_ensemble` members.  The first frame of every run
        is sampled from noise (sample()); every later frame refines each member's latent of the previous frame (refine(), `steps`
        of the T steps, default T // 4), so members stay coherent along a run and cost steps / T of the loop per frame.  More chunks
        put more frames into one pass and break coherence chunks - 1 times.  A run that has ended repeats its last frame, and that
        result is dropped.  With `seed` (instead of `generator`) member e of frame f draws keyed noise (engine.keyed_normal) with key
        f * 2^16 + e, draw 0 when it is sampled and draw 1 when it is refined, so its noise does not depend on `chunks`; its result
        still does, through the warm start it refines.  relax = dict(iterations=..., threshold=...) (either may be left out) relaxes
        every frame's coordinates with relax() before they are stored; the warm starts keep the unrelaxed latents, so relaxing changes
        no frame's sampling.  Returns host float32 [n_frames, num_ensemble, Na, 3]."""
        batches = list(batches)
        steps, runs = trajectory_args(self.T, len(batches), num_ensemble, steps, chunks)
        relax = relax_option(relax)
        if any(b["num_CGs"].numel() != 1 for b in batches) or len({int(b["num_CGs"].sum()) for b in batches}) != 1:
            raise ValueError("backmap_trajectory: every batch must hold one frame, all of the same length")

        def frame_set(p, frames):
            fs = frames_from_batch(batching.merge_batches([batches[f] for f in frames]), info, num_ensemble)
            return self.upload(fs), fs

        return self._trajectory_passes(len(batches), num_ensemble, steps, runs, frame_set, generator, seed, relax=relax)

    def update_coords(self, plan: Plan, fs: FrameSet, ca_full: torch.Tensor):
        """Move a plan uploaded from `fs` (upload()) to new coordinates of the same frames, with no host work: ca_full [fs.F, fs.L+2, 3]
        CUDA float32 on the plan's device, the untrimmed traces (cb2_plan_set_coords).  X, the k-NN graph and h_E0, the 21 A radius
        graph and the IC filters are rebuilt on the device; lengths, residue types, members and topology stay.  Afterwards the host
        fields X, ca_full, csr_row and csr_col of `fs` no longer describe the plan; its slot_atom, frame_of, out_off and num_atoms,
        which decode and residue_motion use, stay valid."""
        if (plan.F, plan.NB, plan.L) != (fs.F, fs.NB, fs.L):
            raise ValueError("the plan was not uploaded from this frame set")
        shape = (fs.F, fs.L + 2, 3)
        if not torch.is_tensor(ca_full) or ca_full.dtype != torch.float32 or tuple(ca_full.shape) != shape:
            raise ValueError(f"ca_full must be a float32 tensor of shape {shape}")
        if ca_full.device != plan.device:
            raise ValueError(f"ca_full must be on {plan.device}")
        plan.set_coords(self.vae, ca_full)

    def backmap_coords(self, ca_full: torch.Tensor, restype: torch.Tensor, info, num_ensemble: int = 1, steps: int = None,
                       chunks: int = 1, generator: torch.Generator = None, seed: int = None, relax: dict = None) -> torch.Tensor:
        """backmap_trajectory for a trajectory given as a coordinate array: ca_full float32 [n_frames, L+2, 3], host or CUDA, the
        coordinate columns of OG_CG_nxyz of every frame (termini included); restype [L+2] integer, its residue ids
        (OG_CG_nxyz[:, 0]); info the topology tuple.  The topology tables are built on the host once; ca_full is uploaded once,
        whole, and every pass, the first included, moves the plan to its frames with update_coords, so the radius graph, X and
        k-NN graph of every frame are built on the device and no batch dict or host graph is needed.  Same passes, arguments (`seed`
        included, and `relax`) and result as backmap_trajectory: host float32 [n_frames, num_ensemble, Na, 3], equal to
        backmap_trajectory on batches of the same frames wherever the caller's graph follows the same 21 A rule (it can differ only
        for a pair at the cutoff)."""
        check_coords_args(ca_full, restype)
        steps, runs = trajectory_args(self.T, ca_full.shape[0], num_ensemble, steps, chunks)
        relax = relax_option(relax)
        return self._coords_passes(ca_full, restype, info, num_ensemble, steps, runs, generator, seed, relax=relax)

    def _coords_passes(self, ca_full: torch.Tensor, restype: torch.Tensor, info, num_ensemble: int, steps: int, runs, generator,
                       seed=None, key_offset: int = 0, relax: dict = None) -> torch.Tensor:
        """The body of backmap_coords for any subset of a trajectory's runs (start, n) (trajectory_chunks order): one plan holds them
        all, only their frames are uploaded, and frame f draws keyed noise with frame key key_offset + f; relax as relax_option
        returns it.  Returns host float32
        [sum n, num_ensemble, Na, 3], the frames of the runs in order."""
        fs = frames_from_coords(ca_full[[start for start, _ in runs]], restype, info, num_ensemble)
        dev = torch.device("cuda", torch.cuda.current_device())
        rows = torch.cat([torch.arange(start, start + n) for start, n in runs])
        ca_dev = ca_full[rows.to(ca_full.device)].to(dev)
        first = torch.tensor([0] + [n for _, n in runs[:-1]]).cumsum(0).to(dev)      # each run's first row of ca_dev
        last = torch.tensor([n - 1 for _, n in runs], device=dev)

        def frame_set(p, frames):                   # rows first + min(p, last) of ca_dev, gathered on the device
            plan = self.upload(fs) if p == 0 else self.plan_for(fs)
            self.update_coords(plan, fs, ca_dev[first + torch.clamp(last, max=p)])
            return plan, fs

        return self._trajectory_passes(rows.numel(), num_ensemble, steps, runs, frame_set, generator, seed, key_offset, relax)

    def _trajectory_passes(self, n_frames: int, num_ensemble: int, steps: int, runs, frame_set, generator, seed=None,
                           key_offset: int = 0, relax: dict = None) -> torch.Tensor:
        """The pass loop of the trajectory methods.  Pass p puts frame start + min(p, n - 1) of every run (start, n) on one plan through
        frame_set(p, frames) -> (plan, fs); pass 0 samples, every later pass refines each member from its own latent of the pass
        before; with `seed` the frame keys are key_offset + the absolute frame indices (member_keys) and the draw is 0 for pass 0, 1
        after.  With `relax` (relax_option's dict) each pass's coordinates are relaxed (Plan.relax) before they are stored; the next
        pass refines the unrelaxed latent.  Results of runs that have ended are dropped.  Returns host float32 [n_frames, num_ensemble, Na, 3] with n_frames the
        frames of all runs, run after run: the whole trajectory when `runs` are all of its runs."""
        if seed is not None and generator is not None:
            raise ValueError("seed draws the noise itself: it excludes generator")
        if n_frames != sum(n for _, n in runs):
            raise ValueError(f"the runs hold {sum(n for _, n in runs)} frames, not {n_frames}")
        first = [sum(n for _, n in runs[:c]) for c in range(len(runs))]         # each run's first output row
        out = None
        res = None
        for p in range(max(n for _, n in runs)):
            frames = [start + min(p, n - 1) for start, n in runs]
            plan, fs = frame_set(p, frames)
            noise = {"generator": generator} if seed is None else \
                {"seed": seed, "keys": member_keys(fs, [key_offset + f for f in frames]), "draw": int(p > 0)}
            if p == 0:
                res = self.sample(plan, fs, **noise)
                Na = int(fs.num_atoms[0])
                out = torch.empty(n_frames, num_ensemble, Na, 3, dtype=torch.float32, device=plan.device)
            else:
                res = self.refine(plan, fs, res["latent"], steps, **noise)
            live = [c for c, (_, n) in enumerate(runs) if p < n]
            xyz = res["xyz"] if relax is None else plan.relax(res["xyz"], relax["threshold"], relax["iterations"])[0]
            xyz = xyz.view(num_ensemble, len(runs), Na, 3)                        # members are ensemble-major: b = e * chunks + c
            out[[first[c] + p for c in live]] = xyz[:, live].transpose(0, 1)
        return out.cpu()

    def _sample(self, plan: Plan, fs: FrameSet, z, step_noise, use_graph: bool, generator, steps: int = None, seed: int = None,
                keys: torch.Tensor = None, draw: int = 0):
        dev = plan.device
        shape = (fs.NB, fs.L, 3)
        noisy = self.sampler == "ddpm" or self.eta != 0
        bufs = self._bufs.get(id(plan))
        if bufs is None:      # persistent buffers: the CUDA graph of the step loop is keyed on these pointers
            bufs = (torch.empty(*shape, device=dev), torch.empty(self.T, *shape, device=dev) if noisy else None)
            self._bufs[id(plan)] = bufs
        x, noise = bufs
        n = self.T if steps is None else steps                          # the loop reads noise slices [0, steps) only
        if seed is not None:              # keyed: slice 0 into x, slices 1 .. n into noise[:n], in place (the graph key stays)
            keys = self._device_keys(plan, fs, keys)
            keyed_normal(seed, keys, fs.L, draw, 0, 1, out=x.unsqueeze(0))
            if noise is not None:
                keyed_normal(seed, keys, fs.L, draw, 1, n, out=noise[:n])
        elif z is not None:
            x.copy_(z, non_blocking=True)
        else:
            torch.randn(*shape, device=dev, generator=generator, out=x)
        if seed is None and noise is not None:
            if step_noise is not None:
                noise.copy_(step_noise, non_blocking=True)
            else:
                torch.randn(n, *shape, device=dev, generator=generator, out=noise[:n])
        plan.sample(x, noise, use_graph)
        idx, zq, ic, xyz = plan.decode(self.vae, x, denorm=True, num_atoms_total=fs.total_atoms)
        return {"latent": x, "idx": idx, "zq": zq, "ic_recon": ic, "xyz": xyz}

    def _device_keys(self, plan: Plan, fs: FrameSet, keys) -> torch.Tensor:
        """keys (default member_keys(fs)) on the plan's device.  The last host keys of a plan stay on the device, so repeated passes
        with the same members make no copy (a copy from pageable memory would synchronise the stream)."""
        keys = member_keys(fs) if keys is None else keys
        if keys.is_cuda:
            return keys.to(plan.device).contiguous()
        cached = self._keys.get(id(plan))
        if cached is None or not torch.equal(cached[0], keys):
            cached = self._keys[id(plan)] = (keys.clone(), keys.to(plan.device).contiguous())
        return cached[1]

    def backmap_host(self, fs: FrameSet, z=None, step_noise=None, generator: torch.Generator = None, seed: int = None,
                     keys: torch.Tensor = None):
        """End-to-end call with HOST inputs and HOST coordinates out (what bench.py's e2e times):
        H2D of the frame set, per-frame precompute, T-step sampling, decode, D2H of [sum Na, 3].  Noise as in sample()."""
        plan = self.upload(fs)
        out = self.sample(plan, fs, z, step_noise, generator=generator, seed=seed, keys=keys)
        host = self._host_xyz.get(fs.total_atoms)
        if host is None:
            host = self._host_xyz[fs.total_atoms] = torch.empty(fs.total_atoms, 3, dtype=torch.float32).pin_memory()
        host.copy_(out["xyz"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host


# ------------------------------------------------------------------------------------------------ multi-GPU
def partition_units(lengths, num_ensemble: int, world: int, k_neighbors: int = 64):
    """Units of the sampling job = (frame, ensemble member), all independent (SURVEY.md section 8e).  Returns, per rank, the
    sorted list of (frame, member) it owns.  Cost of a unit ~ L * min(K, L) edges.  With at least one frame per rank whole
    frames are dealt out (longest-processing-time first), so each frame's k-NN graph / edge features are built once; with
    fewer frames than ranks the units themselves are dealt out and a frame's features are rebuilt on every rank that holds
    one of its members (configs[1] / configs[3]: one frame, members over the GPUs)."""
    F = len(lengths)
    cost = [float(n) * min(int(k_neighbors), int(n)) for n in lengths]
    if F >= world:
        frames = distributed.shard_by_cost([c * num_ensemble for c in cost], world)
        return [[(f, e) for f in fr for e in range(num_ensemble)] for fr in frames]
    units = [(f, e) for f in range(F) for e in range(num_ensemble)]
    parts = distributed.shard_by_cost([cost[f] for f, _ in units], world)
    return [[units[i] for i in p] for p in parts]


def partition_trajectory_units(n_frames, lengths, num_ensemble: int, steps: int, T: int, chunks: int, world: int,
                               k_neighbors: int = 64):
    """Units of a trajectory job = (trajectory t, run c).  Trajectory t (n_frames[t] frames of lengths[t] residues) is split into
    runs = trajectory_chunks(n_frames[t], min(chunks, n_frames[t])), which depend on the job alone, never on `world`.  A run of n
    frames costs L * min(K, L) * num_ensemble * (T + (n - 1) * steps): one full pass, then n - 1 refinements of `steps` steps.  The
    units are dealt out longest-processing-time first (distributed.shard_by_cost).  Returns (runs, parts): runs[t] the [(first
    frame, length)] of trajectory t, parts[r] the (t, c) units of rank r in ascending order (empty when there are fewer units than
    ranks)."""
    if isinstance(chunks, bool) or not isinstance(chunks, numbers.Integral) or chunks < 1:
        raise ValueError(f"chunks must be a positive integer, got {chunks!r}")
    if len(n_frames) != len(lengths):
        raise ValueError(f"{len(n_frames)} frame counts for {len(lengths)} lengths")
    runs = [trajectory_chunks(int(n), min(int(chunks), int(n))) for n in n_frames]
    units = [(t, c) for t in range(len(runs)) for c in range(len(runs[t]))]
    cost = [float(lengths[t]) * min(int(k_neighbors), int(lengths[t])) * num_ensemble * (T + (runs[t][c][1] - 1) * steps)
            for t, c in units]
    return runs, [[units[i] for i in part] for part in distributed.shard_by_cost(cost, world)]


def trajectory_key_offsets(n_frames):
    """Frame-key offsets of a trajectory job: offset_t = the frames of trajectories 0 .. t-1, so frame f of trajectory t has the
    frame key offset_t + f, its index in the whole job.  Refuses a job whose keys would reach 2^47 (member_keys)."""
    offsets, total = [], 0
    for n in n_frames:
        offsets.append(total)
        total += int(n)
    if total > FRAME_KEY_LIMIT:
        raise ValueError(f"the job holds {total} frames in {len(offsets)} trajectories: its frame keys (frame index in the job) "
                         f"must lie in [0, 2^47)")
    return offsets


def group_by_length(frames, lengths, max_frames: int = 32, max_pad: float = 0.12):
    """Frames of one rank -> groups that share a padded plan: longest first, a frame joins the current group while the
    group stays within `max_frames` and its padding (Lmax * n - sum L) / sum L within `max_pad`."""
    order = sorted(frames, key=lambda f: (-lengths[f], f))
    groups, cur, tot = [], [], 0
    for f in order:
        if cur and (len(cur) >= max_frames or (lengths[cur[0]] * (len(cur) + 1) - (tot + lengths[f])) > max_pad * (tot + lengths[f])):
            groups.append(cur)
            cur, tot = [], 0
        cur.append(f)
        tot += lengths[f]
    if cur:
        groups.append(cur)
    return groups


class ShardedBackmapper:
    """The multi-GPU driver of the sampling job (the reference runs loops 1-4 of test.py:413-582 in one process on one
    GPU): every rank holds the whole (host) input, takes its share of the (frame, member) units by cost, back-maps them
    with its own `Backmapper`, and the coordinates are collected on rank 0's host.  No collective on the data path; the
    only communication is that final point-to-point gather."""

    def __init__(self, backmapper, rank: int | None = None, world: int | None = None, max_frames: int = 32, max_pad: float = 0.12):
        r, w, _ = distributed.env_rank_world()
        self.bm, self.rank, self.world = backmapper, (r if rank is None else rank), (w if world is None else world)
        self.max_frames, self.max_pad = max_frames, max_pad
        self._fs_cache = {}

    def plan(self, lengths, num_ensemble: int):
        k = self.bm.k_neighbors if self.bm is not None else 64
        return partition_units(lengths, num_ensemble, self.world, k)

    def local_groups(self, units, lengths):
        """[(frames of the group, frame_of [NB] local indices, [(frame, member)] in member order)] for this rank's units."""
        by_frame = {}
        for f, e in units:
            by_frame.setdefault(f, []).append(e)
        out = []
        for frames in group_by_length(sorted(by_frame), lengths, self.max_frames, self.max_pad):
            members = [(f, e) for f in frames for e in by_frame[f]]
            members.sort(key=lambda fe: (fe[1], frames.index(fe[0])))              # ensemble-major like the single-GPU driver
            out.append((frames, [frames.index(f) for f, _ in members], members))
        return out

    def backmap_local(self, batches, infos, units, lengths, generator=None, seed=None):
        """Back-map this rank's units: {(frame, member): host tensor [Na, 3]}.  With `seed` (instead of `generator`) unit (f, e) draws
        keyed noise with key f * 2^16 + e (unit_keys), f its index in the whole job: what frames_from_batch of the whole job with
        member_keys gives it on one GPU, so its noise does not depend on the world size or on the group it lands in."""
        res = {}
        for frames, frame_of, members in self.local_groups(units, lengths):
            # the padded / CSR form of a group is input-format conversion: done once per group of frames (keyed on the very batch
            # objects), not once per pass
            key = (tuple(id(batches[f]) for f in frames), tuple(frame_of))
            fs = self._fs_cache.get(key)
            if fs is None:
                fs = frames_from_batch(batching.merge_batches([batches[f] for f in frames]), [infos[f] for f in frames], frame_of=frame_of).pin()
                if len(self._fs_cache) >= 64:
                    self._fs_cache.pop(next(iter(self._fs_cache)))
                self._fs_cache[key] = fs
                fs._keep = [batches[f] for f in frames]          # the ids in the key stay valid while the entry lives
            keys = None if seed is None else unit_keys(members)
            host = self.bm.backmap_host(fs, generator=generator, seed=seed, keys=keys)
            for b, fe in enumerate(members):
                o, na = int(fs.out_off[b]), int(fs.num_atoms[frame_of[b]])
                res[fe] = host[o:o + na].clone()
        return res

    def backmap(self, batches, infos, num_ensemble: int, generator=None, _compute=None, seed=None):
        """batches: one reference-schema batch dict per frame (CG_collate of a single frame), infos: its `info` tuple.
        Returns on rank 0 {(frame, member): [Na, 3]} for EVERY unit of the job, on the other ranks None.  With `seed` every unit
        gets the same noise on any number of GPUs (backmap_local).  Its result can still depend on the number of GPUs: the model
        depends on the padded length of the plan a frame is sampled in, and group_by_length groups a rank's frames differently
        for different shares of the job."""
        import torch.distributed as dist
        lengths = [int(b["num_CGs"].sum()) for b in batches]
        n_atoms = [int(i[0].numel()) for i in infos]
        parts = self.plan(lengths, num_ensemble)
        noise = {} if seed is None else {"seed": seed}                  # a compute hook that takes no seed refuses one loudly
        compute = _compute or self.backmap_local
        mine = compute(batches, infos, parts[self.rank], lengths, generator, **noise) if parts[self.rank] else {}
        if self.world == 1 or not (dist.is_available() and dist.is_initialized()):
            return mine
        flat = lambda units, res: torch.cat([res[u] for u in units], 0) if units else torch.zeros(0, 3)
        if self.rank != 0:
            if parts[self.rank]:
                buf = flat(parts[self.rank], mine).contiguous()
                dist.send(buf.cuda() if dist.get_backend() == "nccl" else buf, dst=0)
            return None
        out = dict(mine)
        for r in range(1, self.world):
            if not parts[r]:
                continue
            rows = sum(n_atoms[f] for f, _ in parts[r])
            buf = torch.empty(rows, 3, device="cuda" if dist.get_backend() == "nccl" else "cpu")
            dist.recv(buf, src=r)
            buf, o = buf.cpu(), 0
            for f, e in parts[r]:
                out[(f, e)] = buf[o:o + n_atoms[f]]
                o += n_atoms[f]
        return out

    def backmap_coords_local(self, trajectories, units, runs, offsets, num_ensemble: int, steps: int, generator=None, seed=None,
                             relax=None):
        """Back-map this rank's (trajectory, run) units of a trajectory job: {(t, c): host float32 [n_run, num_ensemble, Na_t, 3]}.
        The local runs of one trajectory share one plan, as `chunks` runs do in Backmapper.backmap_coords, and only their frames are
        uploaded.  With `seed` frame f of trajectory t draws with frame key offsets[t] + f, its index in the whole job.  relax as
        relax_option returns it."""
        by_traj = {}
        for t, c in units:
            by_traj.setdefault(t, []).append(c)
        res = {}
        for t, cs in by_traj.items():
            ca_full, restype, info = trajectories[t]
            xyz = self.bm._coords_passes(ca_full, restype, info, num_ensemble, steps, [runs[t][c] for c in cs], generator, seed,
                                         offsets[t], relax)
            row = 0
            for c in cs:
                n = runs[t][c][1]
                res[(t, c)] = xyz[row:row + n]
                row += n
        return res

    def backmap_coords(self, trajectories, num_ensemble: int = 1, steps: int = None, chunks: int = 1, generator=None, seed=None,
                       _compute=None, relax=None):
        """Backmapper.backmap_coords for a job of trajectories over the ranks.  trajectories: a list of (ca_full [n_t, L_t+2, 3],
        restype [L_t+2], info_t), each what backmap_coords takes; num_ensemble, steps (default T // 4) and chunks apply to every
        trajectory.  Trajectory t is split into min(chunks, n_t) runs, the same on any number of GPUs, and the (t, run) units are
        dealt out by cost (partition_trajectory_units); a rank backmaps its runs of one trajectory in one plan with warm starts.
        Returns on rank 0 a list of host float32 [n_t, num_ensemble, Na_t, 3], one per trajectory in input order; the other ranks send
        their runs to rank 0 one unit at a time and return None.  With no process group (or world 1) a rank returns that list with
        its own runs filled in and the others NaN: the whole result for world 1.
        With `seed`, frame f of trajectory t draws keyed noise with frame key (frames of trajectories before t) + f, so a
        one-trajectory job draws what Backmapper.backmap_coords(seed=) draws.  A trajectory is never padded and its runs do not
        depend on the world size, so the result does not either: bit for bit in the fp32 tier, within the f16 tier's tolerance (its
        MMA tiles sum a row's neighbours in a layout that depends on the row's place in the plan).  With `generator` every rank draws
        from its own generator, and the result depends on the partition.  relax as in Backmapper.backmap_coords: relaxation is per
        member and deterministic, so it keeps the result independent of the world size."""
        import torch.distributed as dist
        trajectories = list(trajectories)
        relax = relax_option(relax)
        if not trajectories:
            raise ValueError("backmap_coords: the job holds no trajectory")
        if seed is not None and generator is not None:
            raise ValueError("seed draws the noise itself: it excludes generator")
        if isinstance(chunks, bool) or not isinstance(chunks, numbers.Integral) or chunks < 1:
            raise ValueError(f"chunks must be a positive integer, got {chunks!r}")
        for t, traj in enumerate(trajectories):
            try:
                if not isinstance(traj, (tuple, list)) or len(traj) != 3:
                    raise ValueError("it must be a tuple (ca_full, restype, info)")
                check_coords_args(traj[0], traj[1])
                steps_t, _ = trajectory_args(self.bm.T, traj[0].shape[0], num_ensemble, steps, min(chunks, traj[0].shape[0]))
            except ValueError as e:
                raise ValueError(f"backmap_coords: trajectory {t}: {e}") from None
        steps = steps_t
        n_frames = [int(ca.shape[0]) for ca, _, _ in trajectories]
        offsets = trajectory_key_offsets(n_frames)
        runs, parts = partition_trajectory_units(n_frames, [int(ca.shape[1]) - 2 for ca, _, _ in trajectories], num_ensemble, steps,
                                                 self.bm.T, chunks, self.world, self.bm.k_neighbors)
        noise = {} if seed is None else {"seed": seed}
        if relax is not None:
            noise["relax"] = relax
        compute = _compute or self.backmap_coords_local
        mine = compute(trajectories, parts[self.rank], runs, offsets, num_ensemble, steps, generator, **noise) if parts[self.rank] else {}
        gather = self.world > 1 and dist.is_available() and dist.is_initialized()
        nccl = gather and dist.get_backend() == "nccl"
        if gather and self.rank != 0:
            for u in parts[self.rank]:                               # partition order, as rank 0 receives them
                dist.send(mine[u].cuda() if nccl else mine[u].contiguous(), dst=0)
            return None
        out = [torch.full((n, num_ensemble, int(info[0].numel()), 3), math.nan) for n, (_, _, info) in zip(n_frames, trajectories)]

        def block(t, c):                                             # the rows of run c in trajectory t's output
            start, n = runs[t][c]
            return out[t][start:start + n]

        for u in parts[self.rank]:
            block(*u).copy_(mine[u])
        if gather:
            for r in range(1, self.world):
                for u in parts[r]:
                    dst = block(*u)
                    if nccl:
                        buf = torch.empty(dst.shape, device="cuda")
                        dist.recv(buf, src=r)
                        dst.copy_(buf)
                    else:
                        dist.recv(dst, src=r)
        return out
