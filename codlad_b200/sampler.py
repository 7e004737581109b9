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

from dataclasses import dataclass, field

import torch

from . import batching, distributed, topology, weights
from .diffusion import create_diffusion
from .engine import DenoiserEngine, Plan, VaeEngine, check_clash_args

VAE_DATA = {"N6": "PED", "K3": "PDB", "K4": "Atlas"}


def clash_pair_totals(counts: torch.Tensor) -> torch.Tensor:
    """Clashing atom pairs per member (int64 [NB]) from per-residue counts [NB, L], where every pair counts for both residues."""
    return counts.sum(1, dtype=torch.int64) // 2


def repair_accept(prev_pairs: torch.Tensor, new_pairs: torch.Tensor) -> torch.Tensor:
    """The acceptance rule of Backmapper.repair, per member: take the resampled latent only if it has fewer clashing pairs."""
    return new_pairs < prev_pairs


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
    csr_row, csr_col = batching.batch_csr(batch["CG_nbr_list"], num, L)
    if frame_of is None:
        frame_of = torch.arange(F, dtype=torch.int32).repeat(num_ensemble)
    frame_of = torch.as_tensor(frame_of, dtype=torch.int32)
    return FrameSet(X, ca_full, cg_z, num.to(torch.int32), csr_row, csr_col, orders, slot_atom, num_atoms, frame_of)


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
        self._host_xyz = {}

    def plan_for(self, fs: FrameSet, keep_debug: bool = False) -> Plan:
        key = (fs.F, fs.NB, fs.L, keep_debug)
        plan = self._plans.get(key)
        if plan is None:
            while len(self._plans) >= self.max_plans:              # a plan owns every buffer of its geometry: keep few of them
                old = self._plans.pop(next(iter(self._plans)))
                self._bufs.pop(id(old), None)
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
               use_graph: bool = True, generator: torch.Generator = None):
        """Device-resident path: returns dict(latent, idx, ic_recon, xyz) of CUDA tensors.
        z [NB,L,3] initial noise, step_noise [T,NB,L,3]; drawn on the device when omitted.  DDIM with eta = 0 uses no
        step noise: `step_noise` is ignored.  Every residue is sampled anew, also after resample() on the same plan."""
        plan.clear_inpaint()
        return self._sample(plan, fs, z, step_noise, use_graph, generator)

    def resample(self, plan: Plan, fs: FrameSet, latent: torch.Tensor, keep: torch.Tensor, z: torch.Tensor = None,
                 step_noise: torch.Tensor = None, generator: torch.Generator = None):
        """Latent inpainting: keep the residues of an earlier pass where keep [NB,L] (bool) is True and sample the others
        anew, conditioned on the kept ones through the denoiser.  latent [NB,L,3] is that pass's normalised latent
        (`sample(...)["latent"]`, which may be passed as is).  Kept rows follow the forward marginal of their latent with the
        fixed draw z and end at it exactly, so they keep their VQ index.  z and step_noise as in sample().  Returns the same
        dict as sample()."""
        shape = (fs.NB, fs.L, 3)
        if not torch.is_tensor(latent) or latent.dtype != torch.float32 or tuple(latent.shape) != shape:
            raise ValueError(f"latent must be a float32 tensor of shape {shape}")
        if not torch.is_tensor(keep) or keep.dtype != torch.bool or tuple(keep.shape) != shape[:2]:
            raise ValueError(f"keep must be a bool tensor of shape {shape[:2]}")
        if latent.device != plan.device or keep.device != plan.device:
            raise ValueError(f"latent and keep must be on {plan.device}")
        plan.set_inpaint(keep, latent, self.diffusion.inpaint_coef_table())      # copies latent before z overwrites its buffer
        return self._sample(plan, fs, z, step_noise, True, generator)

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
               generator: torch.Generator = None):
        """Clash-driven repair of a backmapped sample `out` (the dict of sample() / resample()): each round flags the clashing
        residues (residue_clashes), stops when no member has a clash, and otherwise resamples the flagged residues of every
        member with latent inpainting, fresh noise from `generator`.  Per member the new latent is accepted only when its number
        of clashing pairs went down; otherwise the member keeps its previous latent.  The accepted latents are decoded once at the
        end.  Kept residues keep their latent and VQ index; their coordinates can still move where the IC decoder's radius graph
        reaches a regenerated neighbour.  A round costs one resample pass (one sampling pass plus decode).
        Returns the dict of sample() plus `clashes` (int32 [NB, L], the counts of the returned structure) and `clash_pairs`
        (int64 [rounds run + 1, NB], clashing pairs per member; row 0 is the input's).  The plan is left for plain sample()."""
        if not isinstance(out, dict) or not all(k in out for k in ("latent", "idx", "zq", "ic_recon", "xyz")):
            raise ValueError("out must be the dict returned by sample() or resample()")
        if isinstance(max_rounds, bool) or not isinstance(max_rounds, int) or max_rounds < 0:
            raise ValueError(f"max_rounds must be a non-negative integer, got {max_rounds!r}")
        check_clash_args(threshold, grow, plan.K)
        shape = (fs.NB, fs.L, 3)
        latent = out["latent"]
        if not torch.is_tensor(latent) or latent.dtype != torch.float32 or tuple(latent.shape) != shape or latent.device != plan.device:
            raise ValueError(f"out['latent'] must be a float32 tensor of shape {shape} on {plan.device}")
        counts, keep = self.residue_clashes(plan, fs, out["xyz"], threshold, grow)
        pairs = clash_pair_totals(counts)
        rows = [pairs]
        latent = latent.clone()                  # resample() writes the plan's latent buffer, which out["latent"] may be
        for _ in range(max_rounds):
            if not bool((pairs > 0).any()):
                break
            new = self.resample(plan, fs, latent, keep, generator=generator)
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

    def _sample(self, plan: Plan, fs: FrameSet, z, step_noise, use_graph: bool, generator):
        dev = plan.device
        shape = (fs.NB, fs.L, 3)
        noisy = self.sampler == "ddpm" or self.eta != 0
        bufs = self._bufs.get(id(plan))
        if bufs is None:      # persistent buffers: the CUDA graph of the step loop is keyed on these pointers
            bufs = (torch.empty(*shape, device=dev), torch.empty(self.T, *shape, device=dev) if noisy else None)
            self._bufs[id(plan)] = bufs
        x, noise = bufs
        if z is not None:
            x.copy_(z, non_blocking=True)
        else:
            torch.randn(*shape, device=dev, generator=generator, out=x)
        if noise is not None:
            if step_noise is not None:
                noise.copy_(step_noise, non_blocking=True)
            else:
                torch.randn(self.T, *shape, device=dev, generator=generator, out=noise)
        plan.sample(x, noise, use_graph)
        idx, zq, ic, xyz = plan.decode(self.vae, x, denorm=True, num_atoms_total=fs.total_atoms)
        return {"latent": x, "idx": idx, "zq": zq, "ic_recon": ic, "xyz": xyz}

    def backmap_host(self, fs: FrameSet, z=None, step_noise=None, generator: torch.Generator = None):
        """End-to-end call with HOST inputs and HOST coordinates out (what bench.py's e2e times):
        H2D of the frame set, per-frame precompute, T-step sampling, decode, D2H of [sum Na, 3]."""
        plan = self.upload(fs)
        out = self.sample(plan, fs, z, step_noise, generator=generator)
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

    def backmap_local(self, batches, infos, units, lengths, generator=None):
        """Back-map this rank's units: {(frame, member): host tensor [Na, 3]}."""
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
            host = self.bm.backmap_host(fs, generator=generator)
            for b, fe in enumerate(members):
                o, na = int(fs.out_off[b]), int(fs.num_atoms[frame_of[b]])
                res[fe] = host[o:o + na].clone()
        return res

    def backmap(self, batches, infos, num_ensemble: int, generator=None, _compute=None):
        """batches: one reference-schema batch dict per frame (CG_collate of a single frame), infos: its `info` tuple.
        Returns on rank 0 {(frame, member): [Na, 3]} for EVERY unit of the job, on the other ranks None."""
        import torch.distributed as dist
        lengths = [int(b["num_CGs"].sum()) for b in batches]
        n_atoms = [int(i[0].numel()) for i in infos]
        parts = self.plan(lengths, num_ensemble)
        mine = (_compute or self.backmap_local)(batches, infos, parts[self.rank], lengths, generator) if parts[self.rank] else {}
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
