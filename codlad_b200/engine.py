"""Thin object wrappers over the C ABI: packed models and per-geometry plans.

Everything heavy happens inside libcodlad_b200.so; torch is used for device memory, streams and
host<->device copies only.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers

import numpy as np
import torch

from . import _native as N


def sinusoid_freqs() -> torch.Tensor:
    """exp(-ln(1e4) k / 128), k = 0..127, exactly as the reference forms it
    (models/latent_model.py:59-61), so the CUDA table and a CPU reference share the same bits."""
    import math
    half = 128
    return torch.exp(-math.log(10000) * torch.arange(start=0, end=half, dtype=torch.float32) / half)


def check_clash_args(threshold, grow, K: int):
    """Arguments of the per-residue clash criterion: a finite positive threshold (Angstrom) and 0 <= grow < K (grow = 0 also on a
    decode-only plan, K = 0).  Raises ValueError; touches no device."""
    if isinstance(threshold, bool) or not isinstance(threshold, numbers.Real) or not math.isfinite(threshold) or threshold <= 0:
        raise ValueError(f"threshold must be a finite positive number, got {threshold!r}")
    if isinstance(grow, bool) or not isinstance(grow, numbers.Integral) or grow < 0 or (grow > 0 and grow >= K):
        raise ValueError(f"grow must be an integer in [0, {K}), got {grow!r}")


RELAX_MAX_THRESHOLD = 2.0      # A: above it the repulsion distance reaches the restrained 1-3 geometry of the peptide
RELAX_MAX_ITERATIONS = 100_000


def check_relax_args(threshold, iterations):
    """Arguments of the clash relaxation: threshold (Angstrom) in (0, 2.0] and an integer number of iterations in [0, 10^5].
    Above 2 A the repulsion distance, threshold + 0.2 A, would reach the restrained 1-3 distances of the peptide (about
    2.25-2.45 A), which the relaxation must leave as decoded.  Raises ValueError; touches no device."""
    if isinstance(threshold, bool) or not isinstance(threshold, numbers.Real) or not 0 < threshold <= RELAX_MAX_THRESHOLD:
        raise ValueError(f"threshold must lie in (0, {RELAX_MAX_THRESHOLD}] Angstrom, got {threshold!r}")
    if isinstance(iterations, bool) or not isinstance(iterations, numbers.Integral) or not 0 <= iterations <= RELAX_MAX_ITERATIONS:
        raise ValueError(f"iterations must be an integer in [0, {RELAX_MAX_ITERATIONS}], got {iterations!r}")


def check_start_steps(steps):
    """Argument of Plan.set_start: a non-negative integer (0 = the whole schedule).  Raises ValueError; touches no device."""
    if isinstance(steps, bool) or not isinstance(steps, numbers.Integral) or steps < 0:
        raise ValueError(f"steps must be a non-negative integer, got {steps!r}")


class DenoiserEngine:
    """Packed device copy of an `mpnn_diffusion` state_dict (models/latent_model.py:78-165)."""

    def __init__(self, state_dict: dict, k_neighbors: int = 64):
        N.require_cuda()
        arr, keep = N.tensor_table({k.removeprefix("module."): v for k, v in state_dict.items()})
        freqs = sinusoid_freqs().contiguous()
        h = C.c_void_p()
        N.check(N.lib().cb2_denoiser_create(arr, len(arr), freqs.data_ptr(), int(k_neighbors), C.byref(h)), "denoiser_create")
        self.handle, self.k_neighbors = h, int(k_neighbors)
        del keep

    def close(self):
        if getattr(self, "handle", None) and N is not None and getattr(N, "lib", None) is not None:
            N.lib().cb2_denoiser_destroy(self.handle)
            self.handle = None

    __del__ = close


class VaeEngine:
    """Packed decode-side VQ-VAE state: codebook, map_out, IC decoder (models/vae_model.py:686-839)."""

    def __init__(self, state_dict: dict, mean, std, angle_variant: bool = False):
        N.require_cuda()
        state = dict(state_dict)
        cb = state.get("quantize._codebook.embed")
        if cb is None:
            raise KeyError("state_dict has no 'quantize._codebook.embed'")
        state["quantize._codebook.embed"] = cb.reshape(-1, 3)
        arr, keep = N.tensor_table(state)
        mean = torch.as_tensor(mean, dtype=torch.float32).cpu().contiguous()
        std = torch.as_tensor(std, dtype=torch.float32).cpu().contiguous()
        h = C.c_void_p()
        N.check(N.lib().cb2_vae_create(arr, len(arr), mean.data_ptr(), std.data_ptr(), int(bool(angle_variant)), C.byref(h)),
                "vae_create")
        self.handle, self.angle_variant = h, bool(angle_variant)
        self.codebook_size = cb.reshape(-1, 3).shape[0]
        del keep

    def close(self):
        if getattr(self, "handle", None) and N is not None and getattr(N, "lib", None) is not None:
            N.lib().cb2_vae_destroy(self.handle)
            self.handle = None

    __del__ = close


class Plan:
    """Buffers + CUDA graph for one batch geometry (F frames x L residues, NB members)."""

    def __init__(self, denoiser: DenoiserEngine, F: int, NB: int, L: int, precision: str = "fp32", keep_debug: bool = False):
        self.denoiser = denoiser
        self.F, self.NB, self.L, self.precision = int(F), int(NB), int(L), precision
        h = C.c_void_p()
        N.require_cuda()
        N.check(N.lib().cb2_plan_create(denoiser.handle if denoiser is not None else None, self.F, self.NB, self.L,
                                        N.PRECISION[precision], int(keep_debug), C.byref(h)), "plan_create")
        self.handle = h
        self.K = N.lib().cb2_plan_K(h)
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._lengths = None

    def close(self):
        if getattr(self, "handle", None) and N is not None and getattr(N, "lib", None) is not None:
            N.lib().cb2_plan_destroy(self.handle)
            self.handle = None

    __del__ = close

    @property
    def launches(self) -> int:
        return int(N.lib().cb2_plan_launches(self.handle))

    # -- geometry ------------------------------------------------------------------------------
    def set_frames(self, X, lengths, cg_z, frame_of):
        X = X.to(self.device, torch.float32, non_blocking=True).contiguous()
        lengths = lengths.to(self.device, torch.int32, non_blocking=True).contiguous()
        cg_z = cg_z.to(self.device, torch.int32, non_blocking=True).contiguous()
        frame_of = frame_of.to(self.device, torch.int32, non_blocking=True).contiguous()
        assert X.shape == (self.F, self.L, 3) and cg_z.shape == (self.F, self.L)
        assert lengths.shape == (self.F,) and frame_of.shape == (self.NB,)
        N.check(N.lib().cb2_plan_set_frames(self.handle, N.dptr(X), N.dptr(lengths), N.dptr(cg_z), N.dptr(frame_of), N.stream_ptr()),
                "set_frames")
        self._lengths = lengths
        self._frame_of = frame_of

    def set_topology(self, vae: VaeEngine, ca_full, csr_row, csr_col, orders, slot_atom, out_off):
        ca_full = ca_full.to(self.device, torch.float32, non_blocking=True).contiguous()
        assert ca_full.shape == (self.F, self.L + 2, 3)
        # host or device tensors are both accepted (cudaMemcpyDefault): a batch dict that already lives on the GPU (test.py:487
        # batch_to(device)) is converted on the GPU and never comes back to the host
        csr_row = csr_row.to(torch.int32).contiguous()
        csr_col = csr_col.to(torch.int32).contiguous()
        orders = orders.to(torch.int8).contiguous()
        slot_atom = slot_atom.to(torch.int32).contiguous()
        out_off = out_off.to(torch.int64).contiguous()
        assert csr_row.numel() == self.F * self.L + 1 and orders.numel() == self.F * self.L * 30
        assert slot_atom.numel() == self.F * self.L * 14 and out_off.numel() == self.NB
        N.check(N.lib().cb2_plan_set_topology(self.handle, vae.handle, N.dptr(ca_full), csr_row.data_ptr(), csr_col.data_ptr(),
                                              int(csr_col.numel()), orders.data_ptr(), slot_atom.data_ptr(), out_off.data_ptr(),
                                              N.stream_ptr()), "set_topology")

    def set_coords(self, vae: VaeEngine, ca_full):
        """Move the frames already on the plan to new coordinates, all on the device (cb2_plan_set_coords): ca_full [F, L+2, 3] CUDA
        float32 on the plan's device, the untrimmed traces.  X, the k-NN graph, edge features and h_E0, the radius graph at the VAE's
        cutoff and the IC filters are recomputed from it; lengths, residue types, members and topology stay.  Needs set_topology.
        The step loop's captured graph stays valid."""
        shape = (self.F, self.L + 2, 3)
        if not torch.is_tensor(ca_full) or ca_full.dtype != torch.float32 or tuple(ca_full.shape) != shape:
            raise ValueError(f"ca_full must be a float32 tensor of shape {shape}")
        if ca_full.device != self.device:
            raise ValueError(f"ca_full must be on {self.device}")
        N.check(N.lib().cb2_plan_set_coords(self.handle, vae.handle, N.dptr(ca_full.contiguous()), N.stream_ptr()), "set_coords")

    # -- denoiser --------------------------------------------------------------------------------
    def forward(self, x, t):
        x = x.to(self.device, torch.float32).contiguous()
        t = t.to(self.device, torch.float32).contiguous()
        assert x.shape == (self.NB, self.L, 3) and t.shape == (self.NB,)
        out = torch.empty(self.NB, self.L, 6, device=self.device, dtype=torch.float32)
        N.check(N.lib().cb2_plan_forward(self.handle, N.dptr(x), N.dptr(t), N.dptr(out), N.stream_ptr()), "forward")
        return out

    def forward_partial(self, x, t, stop_after: int):
        """Parity helper: run only the first `stop_after` kernels of forward(); read state with buffer()."""
        x = x.to(self.device, torch.float32).contiguous()
        t = t.to(self.device, torch.float32).contiguous()
        N.check(N.lib().cb2_plan_forward_partial(self.handle, N.dptr(x), N.dptr(t), int(stop_after), N.stream_ptr()), "forward_partial")

    def set_schedule(self, timestep_map, coef):
        t = torch.as_tensor(np.asarray(timestep_map), dtype=torch.float32).contiguous()
        c = torch.as_tensor(np.asarray(coef), dtype=torch.float32).contiguous()
        assert c.shape == (t.numel(), 8)
        N.check(N.lib().cb2_plan_set_schedule(self.handle, t.data_ptr(), c.data_ptr(), int(t.numel()), N.stream_ptr()), "set_schedule")
        self.T = int(t.numel())

    def set_ddim_schedule(self, timestep_map, coef):
        """DDIM schedule: coef = SpacedDiffusion.ddim_coef_table(eta); sample() then applies DDIM updates."""
        t = torch.as_tensor(np.asarray(timestep_map), dtype=torch.float32).contiguous()
        c = torch.as_tensor(np.asarray(coef), dtype=torch.float32).contiguous()
        assert c.shape == (t.numel(), 8)
        N.check(N.lib().cb2_plan_set_ddim_schedule(self.handle, t.data_ptr(), c.data_ptr(), int(t.numel()), N.stream_ptr()),
                "set_ddim_schedule")
        self.T = int(t.numel())

    def sample(self, x, noise=None, use_graph: bool = True):
        """In-place reverse diffusion of x [NB,L,3] with noise [T,NB,L,3] (both CUDA fp32 contiguous).  noise may be None
        on a DDIM schedule with eta = 0 (the C side refuses it otherwise)."""
        assert x.shape == (self.NB, self.L, 3) and (noise is None or noise.shape == (self.T, self.NB, self.L, 3))
        N.check(N.lib().cb2_plan_sample(self.handle, N.dptr(x, torch.float32), N.dptr(noise, torch.float32), int(use_graph), N.stream_ptr()),
                "sample")
        return x

    def set_inpaint(self, keep, x0, q_coef):
        """Latent inpainting for the following sample() calls: the rows where keep [NB,L] (CUDA bool) is True follow the
        normalised latent x0 [NB,L,3] (CUDA fp32), the others are regenerated.  q_coef = SpacedDiffusion.inpaint_coef_table()
        of the plan's schedule.  keep and x0 are copied into plan-owned buffers, so x0 may be the tensor later passed to
        sample(); changing them does not recapture the graph."""
        if not torch.is_tensor(keep) or keep.dtype != torch.bool or tuple(keep.shape) != (self.NB, self.L):
            raise ValueError(f"keep must be a bool tensor of shape {(self.NB, self.L)}")
        if not torch.is_tensor(x0) or x0.dtype != torch.float32 or tuple(x0.shape) != (self.NB, self.L, 3):
            raise ValueError(f"x0 must be a float32 tensor of shape {(self.NB, self.L, 3)}")
        if keep.device != self.device or x0.device != self.device:
            raise ValueError(f"keep and x0 must be on {self.device}")
        q = torch.as_tensor(np.asarray(q_coef), dtype=torch.float32).contiguous()
        if q.dim() != 2 or q.shape[0] < 2 or q.shape[1] != 2:
            raise ValueError("q_coef must be a [T+1, 2] table (SpacedDiffusion.inpaint_coef_table)")
        N.check(N.lib().cb2_plan_set_inpaint(self.handle, N.dptr(keep.to(torch.uint8).contiguous()), N.dptr(x0.contiguous()),
                                             q.data_ptr(), int(q.shape[0]) - 1, N.stream_ptr()), "set_inpaint")

    def set_start(self, steps: int):
        """Partial-noise refinement for the following sample() calls (cb2_plan_set_start): steps = 0 runs the whole schedule;
        1 <= steps <= T runs only respaced steps steps-1 .. 0 and refines the inpainting latent x0 of set_inpaint, which must be
        on.  Every row then starts at the forward marginal of its x0 at that level, with the x passed to sample() as the noise;
        kept rows still end at x0.  noise slices [0, steps) are read.  sample() refuses steps > T or steps without inpainting."""
        check_start_steps(steps)
        N.check(N.lib().cb2_plan_set_start(self.handle, int(steps), N.stream_ptr()), "set_start")

    def clear_inpaint(self):
        """Turn latent inpainting off: sample() regenerates every row again."""
        N.check(N.lib().cb2_plan_set_inpaint(self.handle, None, None, None, 0, N.stream_ptr()), "set_inpaint")

    def run_edge_kernel(self, mode: int, layer: int):
        """Measurement hook: one per-edge kernel on the current state (0 enc node msg, 1 enc edge update, 2 dec msg)."""
        N.check(N.lib().cb2_plan_run_edge_kernel(self.handle, int(mode), int(layer), N.stream_ptr()), "run_edge_kernel")

    def run_stage(self, stage: int, layer: int = 0, vae: "VaeEngine | None" = None, xyz_scratch=None):
        """Measurement hook: one stage of the path on the plan's buffers (see cb2_plan_run_stage in include/codlad_b200.h)."""
        N.check(N.lib().cb2_plan_run_stage(self.handle, vae.handle if vae is not None else None, int(stage), int(layer),
                                           N.dptr(xyz_scratch) if xyz_scratch is not None else None, N.stream_ptr()), "run_stage")

    # -- decode ----------------------------------------------------------------------------------
    def decode(self, vae: VaeEngine, latent, denorm: bool, num_atoms_total: int | None = None, want_ic: bool = True):
        latent = latent.to(self.device, torch.float32).contiguous()
        idx = torch.empty(self.NB, self.L, device=self.device, dtype=torch.int32)
        zq = torch.empty(self.NB, self.L, 3, device=self.device, dtype=torch.float32)
        ic = torch.empty(self.NB, self.L, 13, 3, device=self.device, dtype=torch.float32) if want_ic else None
        xyz = torch.zeros(num_atoms_total, 3, device=self.device, dtype=torch.float32) if num_atoms_total else None
        N.check(N.lib().cb2_plan_decode(self.handle, vae.handle, N.dptr(latent), int(denorm), N.dptr(idx), N.dptr(zq),
                                        N.dptr(ic) if ic is not None else None, N.dptr(xyz) if xyz is not None else None,
                                        N.stream_ptr()), "decode")
        return idx, zq, ic, xyz

    def residue_clashes(self, xyz, threshold: float = 1.2, grow: int = 0):
        """Per-residue clash counts of a decoded sample and the keep mask that resamples the clashing residues
        (cb2_plan_residue_clashes; needs set_topology).  xyz [total atoms, 3] CUDA fp32 as decode() writes it.  Returns
        (counts [NB, L] int32, keep [NB, L] bool): counts[b, i] = atom pairs of residue i with other residues of member b closer
        than `threshold` (peptide bond left out), keep False where residue i or one of its `grow` nearest other residues clashes."""
        if not torch.is_tensor(xyz) or xyz.dtype != torch.float32 or xyz.dim() != 2 or xyz.shape[1] != 3:
            raise ValueError("xyz must be a float32 tensor of shape [total atoms, 3]")
        if xyz.device != self.device:
            raise ValueError(f"xyz must be on {self.device}")
        check_clash_args(threshold, grow, self.K)
        counts = torch.empty(self.NB, self.L, device=self.device, dtype=torch.int32)
        keep = torch.empty(self.NB, self.L, device=self.device, dtype=torch.uint8)
        N.check(N.lib().cb2_plan_residue_clashes(self.handle, N.dptr(xyz.contiguous()), C.c_float(threshold), int(grow), N.dptr(counts),
                                                 N.dptr(keep), N.stream_ptr()), "residue_clashes")
        return counts, keep.view(torch.bool)

    def relax(self, xyz, threshold: float = 1.2, iterations: int = 50):
        """Restrained clash relaxation of a decoded sample (cb2_plan_relax; needs set_topology).  xyz [total atoms, 3] CUDA fp32 as
        decode() writes it; it is not modified.  Returns (xyz_out, max_shift [NB], max_restraint_dev [NB]): the relaxed copy (C-alphas,
        padded and absent rows as given), and per member the largest distance an atom moved and the largest deviation of a restrained
        distance from its input value.  See Backmapper.relax for the objective."""
        if not torch.is_tensor(xyz) or xyz.dtype != torch.float32 or xyz.dim() != 2 or xyz.shape[1] != 3:
            raise ValueError("xyz must be a float32 tensor of shape [total atoms, 3]")
        if xyz.device != self.device:
            raise ValueError(f"xyz must be on {self.device}")
        check_relax_args(threshold, iterations)
        out = xyz.contiguous().clone()
        shift = torch.empty(self.NB, device=self.device, dtype=torch.float32)
        dev = torch.empty(self.NB, device=self.device, dtype=torch.float32)
        N.check(N.lib().cb2_plan_relax(self.handle, N.dptr(out), N.dptr(out), C.c_float(threshold), int(iterations), N.dptr(shift),
                                       N.dptr(dev), N.stream_ptr()), "relax")
        return out, shift, dev

    # -- debug -------------------------------------------------------------------------------------
    def buffer(self, name: str) -> torch.Tensor:
        """Copy of a plan-owned buffer (parity tests)."""
        edge_dtype = torch.float16 if N.PRECISION[self.precision] == 1 else torch.float32
        spec = {
            "nbr_idx": (torch.int32, (self.F, self.L, self.K)), "nbr_dist": (torch.float32, (self.F, self.L, self.K)),
            "E": (torch.float32, (self.F, self.L, self.K, 128)), "hE0": (edge_dtype, (self.F, self.L, self.K, 128)),
            "hE": (edge_dtype, (self.NB, self.L, self.K, 128)), "hV": (torch.float32, (self.NB, self.L, 128)),
            "S": (torch.float32, (self.NB, self.L, 128)), "out6": (torch.float32, (self.NB, self.L, 6)),
            "tc_trace": (torch.int64, (6144,)),
            "relax_partner": (torch.int32, (self.NB, self.L, 14, 16)), "relax_d0": (torch.float32, (self.NB, self.L, 14, 16)),
            "relax_nrep": (torch.int32, (self.NB, self.L, 14)),
        }[name]
        out = torch.empty(spec[1], device=self.device, dtype=spec[0])
        N.check(N.lib().cb2_plan_buffer(self.handle, name.encode(), N.dptr(out), out.numel() * out.element_size(), N.stream_ptr()),
                "plan_buffer")
        return out


# ---- stand-alone kernels ----------------------------------------------------------------------
def knn_topk(X: torch.Tensor, lengths, K: int):
    """CUDA replacement of CA_ProteinFeatures._dist (models/protein_mpnn_utils.py:447-459).
    X [F,L,3] CUDA fp32 -> (D [F,L,K] fp32, idx [F,L,K] int32) sorted by (distance, index)."""
    N.require_cuda()
    X = X.contiguous()
    F, L, _ = X.shape
    D = torch.empty(F, L, K, device=X.device, dtype=torch.float32)
    idx = torch.empty(F, L, K, device=X.device, dtype=torch.int32)
    lp = N.dptr(lengths.to(X.device, torch.int32).contiguous()) if lengths is not None else None
    N.check(N.lib().cb2_knn_topk(N.dptr(X, torch.float32), lp, F, L, int(K), N.dptr(D), N.dptr(idx), N.stream_ptr()), "knn_topk")
    return D, idx


NOISE_MAX_SLICES = 2048      # slice index field of the keyed-noise counter: 11 bits above the 21 of the residue row
NOISE_MAX_L = 1 << 21


def _check_uint(name, v, bits):
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or not 0 <= v < (1 << bits):
        raise ValueError(f"{name} must be an integer in [0, 2^{bits}), got {v!r}")


def check_keyed_normal_args(seed, L, draw, first_slice, n_slices):
    """Scalar arguments of keyed_normal: seed in [0, 2^64), 1 <= L < 2^21, draw in [0, 2^32), slices [first_slice, first_slice +
    n_slices) non-empty within [0, 2048).  Raises ValueError; touches no device."""
    _check_uint("seed", seed, 64)
    _check_uint("draw", draw, 32)
    if isinstance(L, bool) or not isinstance(L, numbers.Integral) or not 1 <= L < NOISE_MAX_L:
        raise ValueError(f"L must be an integer in [1, 2^21), got {L!r}")
    for name, v in (("first_slice", first_slice), ("n_slices", n_slices)):
        if isinstance(v, bool) or not isinstance(v, numbers.Integral):
            raise ValueError(f"{name} must be an integer, got {v!r}")
    if first_slice < 0 or n_slices < 1 or first_slice + n_slices > NOISE_MAX_SLICES:
        raise ValueError(f"slices [{first_slice}, {first_slice + n_slices}) must be non-empty and lie in [0, {NOISE_MAX_SLICES})")


def keyed_normal(seed: int, keys: torch.Tensor, L: int, draw: int, first_slice: int, n_slices: int, out: torch.Tensor = None):
    """Keyed standard normals (cb2_keyed_normal): slices [first_slice, first_slice + n_slices) of every member as float32
    [n_slices, NB, L, 3], written into `out` (CUDA float32 contiguous, that shape) when given.  keys int64 [NB] on the current CUDA
    device, one 64-bit key per member.  Each value depends on (seed, key, draw, slice, row, channel) alone: a member's draws are the
    same bit for bit in any batch, at any padded length, and a partial fill equals those slices of a full one.  Slice 0 is a
    sampling pass's start draw and slice 1 + s the noise of respaced step s."""
    N.require_cuda()
    check_keyed_normal_args(seed, L, draw, first_slice, n_slices)
    dev = torch.device("cuda", torch.cuda.current_device())
    if not torch.is_tensor(keys) or keys.dtype != torch.int64 or keys.dim() != 1 or keys.numel() < 1 or keys.device != dev:
        raise ValueError(f"keys must be a non-empty int64 tensor of shape [NB] on {dev}")
    keys = keys.contiguous()
    shape = (int(n_slices), keys.numel(), int(L), 3)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    elif not torch.is_tensor(out) or out.dtype != torch.float32 or tuple(out.shape) != shape or out.device != dev \
            or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous float32 tensor of shape {shape} on {dev}")
    N.check(N.lib().cb2_keyed_normal(int(seed), N.dptr(keys), shape[1], shape[2], int(draw), int(first_slice), int(n_slices), N.dptr(out),
                                     N.stream_ptr()), "keyed_normal")
    return out


def radius_graph(X: torch.Tensor, lengths, cutoff: float = 21.0):
    """Directed radius graph of every frame on the device (cb2_radius_graph_rows / _fill): X [F,L,3] CUDA fp32, lengths [F] (None =
    all L) -> (row_ptr [F*L+1], col [E]) CUDA int32, the layout of batching.batch_csr(synthetic.radius_graph(...)): a CSR over the
    padded rows with frame-local columns ascending, an edge i -> j when i != j, both are below the frame's length and
    sqrt((dx*dx + dy*dy) + dz*dz) <= cutoff in correctly rounded fp32."""
    N.require_cuda()
    if not torch.is_tensor(X) or X.dtype != torch.float32 or X.dim() != 3 or X.shape[2] != 3 or X.shape[0] < 1 or X.shape[1] < 1:
        raise ValueError("X must be a float32 tensor of shape [F, L, 3] with F, L >= 1")
    if isinstance(cutoff, bool) or not isinstance(cutoff, numbers.Real) or not math.isfinite(cutoff) or cutoff < 0:
        raise ValueError(f"cutoff must be a finite non-negative number, got {cutoff!r}")
    X = X.contiguous()
    F, L, _ = X.shape
    if lengths is None:
        lengths = torch.full((F,), L, dtype=torch.int32, device=X.device)
    lengths = torch.as_tensor(lengths).to(X.device, torch.int32).contiguous()
    if lengths.shape != (F,):
        raise ValueError(f"lengths must have shape {(F,)}")
    row_ptr = torch.empty(F * L + 1, device=X.device, dtype=torch.int32)
    N.check(N.lib().cb2_radius_graph_rows(N.dptr(X), N.dptr(lengths), F, L, C.c_float(cutoff), N.dptr(row_ptr), N.stream_ptr()),
            "radius_graph_rows")
    col = torch.empty(int(row_ptr[-1]), device=X.device, dtype=torch.int32)
    if col.numel() == 0:
        return row_ptr, col
    N.check(N.lib().cb2_radius_graph_fill(N.dptr(X), N.dptr(lengths), F, L, C.c_float(cutoff), N.dptr(row_ptr), N.dptr(col),
                                          N.stream_ptr()), "radius_graph_fill")
    return row_ptr, col
