#!/usr/bin/env python
"""bench.py -- backmapped residues/sec of the reverse latent-diffusion sampling path.

One "step" = one pass of the whole hot path over one batch of synthetic input: BASELINE.json configs[1],
a PED-like 300-residue protein, N6 decoder, 100 respaced DDPM steps, num_ensemble = 10 -> 3000 backmapped
residues per rank per step (k-NN graph + edge features once per frame, 100 x denoiser forward + p_sample,
de-normalise, VQ lookup, IC decoder, ic_to_xyz).  At N > 1 every rank samples its own protein (weak scaling,
no collective on the data path; SURVEY.md section 8e).

    python bench.py --gpus N --steps K --warmup W [--precision f16|fp32] [--impl reference] [--dump-outputs DIR]

`--dump-outputs DIR` writes what rank 0's last timed step returned (sampler.Backmapper.sample: latent, idx, zq, ic_recon, xyz) as
DIR/<name>.npy, so that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.

prints ONE JSON line (rank 0):
  value         device-resident throughput (CUDA events, max over ranks, L2 flushed between timed steps)
  e2e           the same metric through the public host API (pinned host inputs -> host coordinates)
  e2e_dropin    the same pass driven through the reference's own call surface (INTEGRATION.md section 1)
  roofline      the dominant kernel (encoder edge update) timed alone with CUDA events, against the measured tensor peak
  roofline_all  every kernel of the path, cold (L2 flushed) and warm, against the peak that bounds it
  scale_checks  the SHARDED product driver (sampler.ShardedBackmapper) on BASELINE configs[2] (256 ragged Atlas-like
                proteins, fixed total: strong scaling over the ranks) and configs[3] (32 members of one 2000-residue frame)
  cpu_baseline  the CPU oracle port on the host cores, bounded samples (what each sample was is stated)
`--impl reference` times that CPU port as the reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (which may be read-only)

import torch  # noqa: E402

METRIC = "backmapped residues/sec (100-step, 10-ensemble)"
UNIT = "residues/s"
L_RES, ENSEMBLE, T_STEPS = 300, 10, 100
WORKLOAD = "configs[1]: PED-like 300-residue IDP, N6, 100-step latent sampling, num_ensemble=10"
# The bench line is configs[1] (`--workload c2`, the configuration the metric is quoted on).  c3 / c4 are BASELINE.json's larger
# configurations at their per-GPU shard size, runnable with the same harness (not bench lines); the sharded product driver runs
# the full configs[2] / configs[3] jobs inside `scale_checks`.
WORKLOADS = {
    "c2": dict(desc=WORKLOAD, L=300, frames=1, ensemble=10, k=64, compact=0.0, vae="N6"),
    "c3": dict(desc="configs[2] per-GPU shard: 32 Atlas-like proteins x 500 residues, K4 decoder, 100 steps, num_ensemble=1",
               L=500, frames=32, ensemble=1, k=64, compact=0.002, vae="K4"),
    "c4": dict(desc="configs[3]: one Atlas-like 2000-residue frame, K4 decoder, k_neighbors=48, 100 steps, 32 members over the GPUs",
               L=2000, frames=1, ensemble=32, k=48, compact=0.002, vae="K4"),
}
C3_JOB = dict(proteins=256, lmin=300, lmax=700, compact=0.002, seed=7300)          # mean length 500 -> ~128 k residues in total

# canonical algorithmic work per edge of the three per-edge kernels (SURVEY.md section 8d): GEMM flops only
EDGE_FLOPS = {0: 2 * 2 * 128 * 128, 1: 2 * 3 * 128 * 128, 2: 2 * 2 * 128 * 128}
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # ALU-bound kernels have no measured peak: nominal FFMA rate, labelled as such
DUMP_LIMIT = 64 << 20                                      # bytes written by --dump-outputs, all arrays together


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 6:
                continue
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except ValueError:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out: dict, path: str):
    """CUDA tensors -> path/<name>.npy: floating point as float32, integer indices as float64 (exact).  When the arrays
    together would exceed DUMP_LIMIT, each keeps the same fixed, seeded sample of its rows (same shapes -> same rows)."""
    import numpy as np
    arrays = {k: v.detach().cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64)
              for k, v in out.items() if v is not None}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT:
            rows = np.random.default_rng(0).choice(a.shape[0], max(1, a.shape[0] * DUMP_LIMIT // total), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(path, name + ".npy"), a)


def _workload(rank: int, name: str = "c2", world: int = 1):
    """Synthetic protein(s) of this rank + host FrameSet (SURVEY.md section 8d generators)."""
    from codlad_b200 import sampler, synthetic
    w = WORKLOADS[name]
    if w["frames"] == 1:
        prot = synthetic.make_protein(w["L"], 1, seed=1002 + (rank if name == "c2" else 0), compact=w["compact"])
        batch = synthetic.collate(prot)
        ens = w["ensemble"] if name == "c2" else max(1, w["ensemble"] // world)      # c4 shards its members over the ranks
        return prot, batch, sampler.frames_from_batch(batch, prot.info, ens)
    prots = [synthetic.make_protein(w["L"], 1, seed=3000 + rank * w["frames"] + i, compact=w["compact"]) for i in range(w["frames"])]
    batch = synthetic.collate_many(prots)
    return prots[0], batch, sampler.frames_from_batch(batch, [p.info for p in prots], w["ensemble"])


# ------------------------------------------------------------------------------------------------ CPU port timing
def _cpu_setup(threads):
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    torch.set_grad_enabled(False)
    return threads


def cpu_port_sample(denoiser_steps: int = 3, threads: int | None = None):
    """Times the CPU oracle (oracle/restate.py, a restatement of the reference's PyTorch path) on the full
    configs[1] batch for `denoiser_steps` denoiser+p_sample steps + graph/features + one decode + one ic_to_xyz and
    extrapolates the homogeneous steps to 100 (SURVEY.md section 8d / BASELINE.md section 3).  The reference
    itself is Python with absent third-party deps and cannot travel to the GPU box, hence kind = "port"."""
    from codlad_b200 import synthetic, weights
    from oracle import restate as R
    threads = _cpu_setup(threads)
    prot, batch, _ = _workload(0)
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    X = prot.ca_full[:, 1:-1].expand(ENSEMBLE, -1, -1).contiguous()
    zz = prot.restype_full[1:-1][None].expand(ENSEMBLE, -1).contiguous()
    mask = torch.ones(ENSEMBLE, L_RES, dtype=torch.bool)
    x = synthetic.latent_noise((ENSEMBLE, L_RES, 3), 1)
    noise = synthetic.latent_noise((denoiser_steps, ENSEMBLE, L_RES, 3), 2)
    sch = R.respaced_schedule(T_STEPS)
    t0 = time.perf_counter()
    g = R.edge_embedding(dsd, X[:1], mask[:1].int(), 64)           # once per frame (hoisted, like the CUDA path)
    t_graph = time.perf_counter() - t0
    graph = tuple(v.expand(ENSEMBLE, *v.shape[1:]).contiguous() for v in (g[0], g[3]))
    R.denoiser_forward(dsd, x, torch.full((ENSEMBLE,), 999), X, zz, mask, 64, graph=graph)      # warm-up
    t0 = time.perf_counter()
    for s in range(denoiser_steps):
        step = T_STEPS - 1 - s
        tt = torch.full((ENSEMBLE,), int(sch["timestep_map"][step]))
        out = R.denoiser_forward(dsd, x, tt, X, zz, mask, 64, graph=graph)
        x = R.p_sample_update(x, out, step, noise[s], sch)
    t_step = (time.perf_counter() - t0) / denoiser_steps
    mean, std = (torch.tensor(v) for v in weights.LATENT_STATS[("N6", "PED")])
    rep = lambda t: torch.cat([t] * ENSEMBLE, 0)
    nbr = torch.cat([batch["CG_nbr_list"] + e * L_RES for e in range(ENSEMBLE)], 0)
    t0 = time.perf_counter()
    ic, _ = R.latent_decode(vsd, x * std + mean, mask, rep(batch["CG_nxyz"][:, 0].long()), rep(batch["CG_nxyz"][:, 1:]), nbr,
                            torch.full((ENSEMBLE,), L_RES), False)
    og = batch["OG_CG_nxyz"].reshape(1, L_RES + 2, 4).expand(ENSEMBLE, -1, -1)
    R.ic_to_xyz(og, ic.reshape(ENSEMBLE, L_RES, 13, 3), prot.info)
    t_dec = time.perf_counter() - t0
    total = t_graph + T_STEPS * t_step + t_dec
    return {
        "value": L_RES * ENSEMBLE / total, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": (f"full configs[1] batch (10x300): graph+features once ({t_graph:.2f}s) + {denoiser_steps} denoiser+p_sample steps "
                   f"({t_step:.2f}s each, extrapolated x{T_STEPS}) + 1 VQ/decode/ic_to_xyz ({t_dec:.2f}s); undoubled batch, "
                   f"features hoisted (the reference as shipped doubles the batch and recomputes features per step)"),
        "seconds_per_pass_extrapolated": total,
    }


def cpu_anchor_c1(threads: int | None = None, shipped_steps: int = 10):
    """configs[0] (1 x 64 residues, ensemble 1) on the CPU port, run IN FULL (100 steps, nothing extrapolated), and the same
    configuration the way the reference driver ships it (test.py:505,533 doubles the batch and throws half away;
    latent_model.py:208 recomputes the k-NN graph and edge features at every step) for `shipped_steps` steps."""
    from codlad_b200 import synthetic, weights
    from oracle import restate as R
    threads = _cpu_setup(threads)
    L = 64
    prot = synthetic.make_protein(L, 1, seed=1001)
    batch = synthetic.collate(prot)
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    X = prot.ca_full[:, 1:-1].contiguous()
    zz = prot.restype_full[1:-1][None].contiguous()
    mask = torch.ones(1, L, dtype=torch.bool)
    z0 = synthetic.latent_noise((1, L, 3), 2001)
    noises = synthetic.latent_noise((T_STEPS, 1, L, 3), 3001)
    sch = R.respaced_schedule(T_STEPS)
    mean, std = (torch.tensor(v) for v in weights.LATENT_STATS[("N6", "PED")])

    def decode(lat):
        ic, _ = R.latent_decode(vsd, lat * std + mean, mask, batch["CG_nxyz"][:, 0].long(), batch["CG_nxyz"][:, 1:], batch["CG_nbr_list"],
                                batch["num_CGs"], False)
        return R.ic_to_xyz(batch["OG_CG_nxyz"].reshape(-1, L + 2, 4), ic.reshape(1, L, 13, 3), prot.info)

    R.denoiser_forward(dsd, z0, torch.full((1,), 999), X, zz, mask, 64)                       # warm-up
    t0 = time.perf_counter()
    decode(R.sample_loop(dsd, z0, X, zz, mask, noises, sch))                                  # hoisted graph, undoubled: all 100 steps
    t_full = time.perf_counter() - t0
    X2, z2, m2 = X.expand(2, -1, -1).contiguous(), zz.expand(2, -1).contiguous(), mask.expand(2, -1).contiguous()
    x = torch.cat([z0, z0], 0)
    t0 = time.perf_counter()
    for s in range(shipped_steps):
        step = T_STEPS - 1 - s
        out = R.denoiser_forward(dsd, x, torch.full((2,), int(sch["timestep_map"][step])), X2, z2, m2, 64)      # graph rebuilt inside
        x = R.p_sample_update(x, out, step, torch.cat([noises[s], noises[s]], 0), sch)
    t_ship_step = (time.perf_counter() - t0) / shipped_steps
    t0 = time.perf_counter()
    decode(x[:1])
    t_dec = time.perf_counter() - t0
    shipped_total = T_STEPS * t_ship_step + t_dec
    return {
        "config": "configs[0]: 1 x 64 residues, N6, 100 steps, num_ensemble=1", "unit": UNIT, "cores": threads, "kind": "port",
        "value": L / t_full, "seconds_per_pass": t_full, "sample": "the whole pass, nothing extrapolated (un-doubled batch, features hoisted)",
        "as_shipped": {"value": L / shipped_total, "seconds_per_pass_extrapolated": shipped_total,
                       "sample": f"doubled batch + graph/features recomputed per step: {shipped_steps} steps of {t_ship_step:.3f}s extrapolated x{T_STEPS} "
                                 f"+ 1 decode ({t_dec:.2f}s)"},
    }


def run_reference(args):
    """`--impl reference`: the CPU port on all host threads; each step is the bounded sample above (3 denoiser steps)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_port_sample(denoiser_steps=3)
        if i >= args.warmup:
            vals.append(r)
    v = sum(x["value"] for x in vals) / len(vals)
    ms = 1e3 * sum(x["seconds_per_pass_extrapolated"] for x in vals) / len(vals)
    cb = dict(vals[-1]); cb["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "CPU port of the reference path (oracle/restate.py); 100-step pass extrapolated from a bounded sample"},
        "cpu_baseline": cb, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------ evaluation-step kernel
def run_metrics(args):
    """`--workload metrics`: the evaluation-step kernel (cb2_eval_bond_graphs, SURVEY.md section 8f-4) on the ensemble configs[1]
    produces, with the CPU oracle port of the reference's eval_sample_qualities timed beside it.  Not the bench line."""
    from codlad_b200 import metrics, sampler, synthetic, weights
    torch.set_grad_enabled(False)
    prot = synthetic.make_protein(L_RES, 1, seed=1002)
    fs = sampler.frames_from_batch(synthetic.collate(prot), prot.info, ENSEMBLE)
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=10, precision=args.precision)
    xyz = bm.sample(bm.upload(fs), fs, generator=torch.Generator(device="cuda").manual_seed(1))["xyz"]
    na = int(fs.num_atoms[0])
    num = [na] * ENSEMBLE
    ref = xyz[:na].repeat(ENSEMBLE, 1).contiguous()              # every member against member 0
    z = torch.tensor([7, 6, 6, 8, 6, 6, 16, 8, 1], dtype=torch.int64).repeat(xyz.shape[0] // 9 + 1)[:xyz.shape[0]].cuda()
    for _ in range(max(args.warmup, 3)):
        metrics.bond_graph_stats(ref, xyz, z, num)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.steps
    a.record()
    for _ in range(reps):
        counts, _ = metrics.bond_graph_stats(ref, xyz, z, num)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    from oracle import restate as R                               # CPU baseline leg
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    c_ref, _ = R.sample_quality_stats(ref.cpu(), xyz.cpu(), z.cpu(), num)
    cpu_s = time.perf_counter() - t0
    print(json.dumps({"metric": "bond-graph comparisons (structures scored per second)", "value": ENSEMBLE / (ms * 1e-3), "unit": "structures/s",
                      "structures": ENSEMBLE, "atoms_per_structure": na, "gpu_ms_per_call": ms, "atom_pairs_per_s": 2 * ENSEMBLE * na * na / (ms * 1e-3),
                      "cpu_baseline": {"value": ENSEMBLE / cpu_s, "unit": "structures/s", "cores": os.cpu_count(), "kind": "port",
                                       "sample": "the same 10 structures, oracle.restate.sample_quality_stats"},
                      "counts_equal_oracle": bool(torch.equal(counts.cpu(), c_ref)),
                      "note": "gpu_ms_per_call is the public call (input checks, one small H2D copy of the offsets, two kernels)"}))


# ------------------------------------------------------------------------------------------------ train_latent step (configs[4])
def run_train(args):
    """`--workload c5`: BASELINE configs[4] -- the train_latent step (denoiser forward + backward in train mode with the reference's
    dropout 0.6, DDP gradient all-reduce over NCCL, clip + AdamW + EMA) on a synthetic PED-like batch of 128 proteins of ragged length
    U[60, 400], global batch fixed (per-rank batch 128 / world, train_latent.py:54).  Not the bench line (that is the sampling path)."""
    from codlad_b200 import distributed as D, synthetic, train, weights
    from codlad_b200.diffusion import create_diffusion
    rank, world, local = D.env_rank_world()
    torch.cuda.set_device(local)
    D.init_from_env("nccl", local)
    dev = torch.device("cuda", local)
    B_total, micro = 128, args.micro_batch
    rnd = random.Random(5000)
    lens = [rnd.randint(60, 400) for _ in range(B_total)]
    per = B_total // world
    mine = sorted(range(rank * per, (rank + 1) * per), key=lambda i: -lens[i])            # padded per micro-batch: group similar lengths
    prots = {i: synthetic.make_protein(lens[i], 1, seed=5100 + i) for i in mine}
    groups = [mine[k:k + micro] for k in range(0, len(mine), micro)]
    batches = [synthetic.collate_many([prots[i] for i in g]) for g in groups]
    gen = torch.Generator().manual_seed(77 + rank)
    data = []
    for g in groups:
        Lm = max(lens[i] for i in g)
        data.append((torch.randn(len(g), Lm, 3, generator=gen), torch.randint(0, 1000, (len(g),), generator=gen)))
    tr = train.DenoiserTrainer(weights.init_denoiser_state(0), lr=1e-4, gemm=args.train_gemm)
    diffusion = create_diffusion("")
    dgen = torch.Generator(device=dev).manual_seed(5 + rank)

    def one_step():
        loss = 0.0
        for k, (g, b, (x1, t)) in enumerate(zip(groups, batches, data)):
            last = k == len(groups) - 1
            _, l = tr.train_step(diffusion, x1, t, b, dropout_p=0.6, generator=dgen, zero=(k == 0), loss_weight=len(g) / per,
                                 do_allreduce=last, do_step=last)
            loss += l * len(g) / per
        return loss

    for _ in range(max(1, min(args.warmup, 2))):
        one_step()
    D.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    losses = []
    for a, b in ev:
        a.record()
        losses.append(one_step())                       # device scalars: nothing inside a step waits for the GPU
        b.record()
    D.barrier()
    losses = [float(v) for v in losses]
    ms = D.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) / args.steps, dev)
    residues = sum(lens)
    padded = D.gather_counts(sum(max(lens[i] for i in g) * len(g) for g in groups), dev)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import restate as R
        threads = _cpu_setup(None)
        torch.set_grad_enabled(True)
        ids = mine[-2:]                                                                  # the two shortest proteins of the batch
        Lm = max(lens[i] for i in ids)
        X = torch.zeros(2, Lm, 3); z = torch.zeros(2, Lm, dtype=torch.int64)
        for q, i in enumerate(ids):
            X[q, :lens[i]] = prots[i].ca_full[0, 1:-1]; z[q, :lens[i]] = prots[i].restype_full[1:-1]
        mask = torch.arange(Lm)[None] < torch.tensor([lens[i] for i in ids])[:, None]
        leaves = {k: v.clone().requires_grad_(True) for k, v in weights.init_denoiser_state(0).items()}
        t0 = time.perf_counter()
        out = R.denoiser_forward(leaves, torch.randn(2, Lm, 3), torch.tensor([500, 10]), X, z, mask, 64)
        (out ** 2).mean().backward()
        cpu_s = time.perf_counter() - t0
        torch.set_grad_enabled(False)
        cpu = {"value": sum(lens[i] for i in ids) / cpu_s, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"torch.autograd through the CPU oracle's forward, 2 proteins ({[lens[i] for i in ids]} residues), one forward + backward, no optimiser"}
    if rank == 0:
        edges = sum(padded) * 64
        flops = 3 * (884736 * edges + 2.16e6 * sum(padded))            # forward (canonical, SURVEY 8d) + two gradient GEMMs per linear layer
        print(json.dumps({
            "metric": "train_latent residues/sec (denoiser fwd+bwd, global batch 128, DDP all-reduce, AdamW+EMA)", "value": residues / (ms * 1e-3),
            "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "tf32 (tcgen05 kind::tf32, fp32 accumulate and storage)" if args.train_gemm == "tf32" else "f32 (SIMT GEMM)", "data": "synthetic",
            "config": {"workload": "configs[4]: train_latent denoiser fwd+bwd, batch 128, PED-like ragged lengths U[60,400], dropout 0.6, DDP NCCL all-reduce",
                       "per_rank_batch": per, "micro_batch": micro, "padded_residues_per_rank": padded, "residues": residues},
            "loss": losses, "grad_norm": tr.grad_norm(), "achieved_tflops": flops / (ms * 1e-3) / 1e12,
            "fp32_nominal_peak_tflops": FP32_NOMINAL_TFLOPS * world, "tf32_nominal_dense_peak_tflops": 1130.0 * world, "cpu_baseline": cpu,
        }))
    D.shutdown()


# ------------------------------------------------------------------------------------------------ per-kernel rooflines
def _time_stage(fn, flush, reps=10):
    """(cold us, warm us) of one launch: cold = L2 flushed before every launch, warm = back to back."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    cold = 0.0
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        cold += a.elapsed_time(b)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(2 * reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return cold / reps * 1e3, a.elapsed_time(b) / (2 * reps) * 1e3


def roofline_all(plan, bm, fs, flush, peaks, precision, traffic):
    """One entry per kernel of the path (SURVEY.md section 8d): algorithmic work / measured launch time against the peak that bounds it.
    `launches_per_pass` x `us_warm` adds up to the pass; kernels that run once per frame / once per pass matter little at configs[1]
    and much at configs[2] (32 new frames per pass)."""
    E = fs.NB * fs.L * plan.K                 # edges per step-loop launch
    FE = fs.F * fs.L * plan.K                 # edges per frame-level launch
    Nn, Fn = fs.NB * fs.L, fs.F * fs.L
    DE = int(fs.csr_col.numel()) * (fs.NB // fs.F)      # directed radius-graph edges seen by the IC decoder (per member)
    xyz = torch.zeros(fs.total_atoms, 3, device=plan.device)
    es = 2 if precision == "f16" else 4
    T = T_STEPS
    spec = [
        # name, fn, bound, flops, bytes, launches per pass
        ("edge message, encoder (edge kernel mode 0)", lambda: plan.run_stage(0, 1), "tensor", EDGE_FLOPS[0] * E, 128 * es * E, 3 * T),
        ("edge update, encoder (edge kernel mode 1)", lambda: plan.run_stage(1, 1), "tensor", EDGE_FLOPS[1] * E, 2 * 128 * es * E, 3 * T),
        ("edge message, decoder (edge kernel mode 2)", lambda: plan.run_stage(2, 1), "tensor", EDGE_FLOPS[2] * E, 128 * es * E, 3 * T),
        ("node update, encoder layer", lambda: plan.run_stage(3, 1), "tensor", 393216 * Nn, (128 * 4 * 3 + 2 * 256 * 2) * Nn, 3 * T),
        ("node update, decoder layer", lambda: plan.run_stage(3, 4), "tensor", 327680 * Nn, (128 * 4 * 3 + 256 * 2) * Nn, 2 * T),
        ("node update + FinalLayer + p_sample", lambda: plan.run_stage(3, 5), "tensor", 327680 * Nn, (128 * 4 * 2 + 36) * Nn, T),
        ("k-NN graph", lambda: plan.run_stage(4), "alu", 8 * fs.L * fs.L * fs.F, (12 + 8 * plan.K) * Fn, 1),
        ("edge featuriser", lambda: plan.run_stage(5), "tensor", 75520 * FE, 128 * es * FE, 1),
        ("IC distance filters", lambda: plan.run_stage(9, 0, bm.vae), "hbm", (15 * 20 + 4 * 2 * 15 * 40) * int(fs.csr_col.numel()), 4 * 40 * 4 * int(fs.csr_col.numel()), 1),
        ("de-normalise + VQ lookup + map_out", lambda: plan.run_stage(6, 0, bm.vae), "alu", 36864 * Nn, (12 + 4 + 12 + 160) * Nn, 1),
        ("IC decoder (messages + heads)", lambda: plan.run_stage(7, 0, bm.vae), "hbm", 4 * 80 * DE + 60000 * Nn, 4 * (160 + 160) * DE + 4 * 39 * Nn, 1),
        ("ic_to_xyz", lambda: plan.run_stage(8, 0, bm.vae, xyz), "hbm", 13 * 120 * Nn, 528 * Nn, 1),
    ]
    out = []
    for name, fn, bound, flops, nbytes, per_pass in spec:
        cold, warm = _time_stage(fn, flush)
        tf, gbs = flops / (cold * 1e-6) / 1e12, nbytes / (cold * 1e-6) / 1e9
        if bound == "tensor":
            ach, peak, unit = tf, peaks["tflops_burst"], "TFLOP/s"
        elif bound == "hbm":
            ach, peak, unit = gbs, peaks["hbm_gbs"], "GB/s"
        else:
            ach, peak, unit = tf, FP32_NOMINAL_TFLOPS, "TFLOP/s (fp32 ALU, NOMINAL peak: no measured ALU figure)"
        out.append({"kernel": name, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                    "us_per_launch": cold, "us_per_launch_l2_resident": warm, "frac_l2_resident": ach / peak * cold / warm,
                    "flops_per_launch": flops, "algorithmic_bytes_per_launch": nbytes, "hbm_gbs_algorithmic": gbs,
                    "launches_per_pass": per_pass, "traffic": (traffic or {}).get(name)})
    return out


# ------------------------------------------------------------------------------------------------ sharded product driver
def _c3_job():
    """BASELINE configs[2] as ONE job: 256 'Atlas-like' proteins (compact random walks, ragged lengths U[300, 700], mean 500)."""
    from codlad_b200 import synthetic
    rnd = random.Random(C3_JOB["seed"])
    lens = [rnd.randint(C3_JOB["lmin"], C3_JOB["lmax"]) for _ in range(C3_JOB["proteins"])]
    prots = [synthetic.make_protein(n, 1, seed=C3_JOB["seed"] + 1 + i, compact=C3_JOB["compact"]) for i, n in enumerate(lens)]
    return prots


def scale_checks(args, D, dev, rank, world):
    """Strong scaling of the sharded driver: a FIXED job split over the ranks by cost, coordinates gathered on rank 0's host.
    Timed on every rank with CUDA events around its own share (H2D, precompute, 100 steps, decode, D2H), max over ranks; the
    wall clock including the final host gather is reported beside it."""
    from codlad_b200 import sampler, synthetic, weights
    out = {}
    jobs = []
    if args.scale in ("all", "c3"):
        prots = _c3_job()
        jobs.append(("configs[2]", "256 Atlas-like proteins, ragged lengths U[300,700] (weakly compacted walk, pull 0.002), K4 decoder, k=64, 100 steps, num_ensemble=1",
                     prots, 1, 64))
    if args.scale in ("all", "c4"):
        jobs.append(("configs[3]", "one Atlas-like 2000-residue frame (weakly compacted walk, pull 0.003), K4 decoder, k_neighbors=48, 100 steps, 32 members",
                     [synthetic.make_protein(2000, 1, seed=1014, compact=0.003)], 32, 48))
    for key, desc, prots, ens, k in jobs:
        batches = [synthetic.collate(p) for p in prots]
        infos = [p.info for p in prots]
        lengths = [p.L for p in prots]
        bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0, True, ("K4", "Atlas")), "K4", k_neighbors=k,
                                num_sampling_steps=T_STEPS, precision=args.precision, max_plans=16)
        sb = sampler.ShardedBackmapper(bm, rank, world)
        parts = sb.plan(lengths, ens)
        cost = [sum(lengths[f] * min(k, lengths[f]) for f, _ in p) for p in parts]
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        res = sb.backmap(batches, infos, ens, generator=gen)                      # warm-up: plans, graphs
        n_units = D.gather_counts(len(parts[rank]), dev)
        passes, ms_dev, ms_wall = max(1, args.scale_passes), 0.0, 0.0
        for _ in range(passes):
            D.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            mine = sb.backmap_local(batches, infos, parts[rank], lengths, gen) if parts[rank] else {}
            b.record()
            torch.cuda.synchronize()
            ms_dev += D.max_over_ranks(a.elapsed_time(b), dev)
            res = sb.backmap(batches, infos, ens, generator=gen, _compute=lambda *_a: mine)      # the gather alone (compute re-used)
            D.barrier()
            ms_wall += D.max_over_ranks((time.perf_counter() - t0) * 1e3, dev)
        residues = sum(lengths) * ens
        groups = sb.local_groups(parts[rank], lengths)
        pad = sum(max(lengths[f] for f in g[0]) * len(g[1]) for g in groups) / max(1, sum(lengths[f] for f, _ in parts[rank]))
        if rank == 0:
            atoms = sum(int(v.shape[0]) for v in res.values())
            out[key] = {"workload": desc, "scaling": "strong", "residues": residues, "units": sum(n_units), "units_per_rank": n_units,
                        "ms_per_pass": ms_dev / passes, "value": residues / (ms_dev / passes * 1e-3), "unit": UNIT,
                        "ms_per_pass_wall_with_host_gather": ms_wall / passes, "atoms_gathered_on_rank0": atoms,
                        "cost_imbalance_max_over_mean": max(cost) / (sum(cost) / len(cost)), "padding_factor_rank0": pad,
                        "plans_rank0": len(groups), "passes": passes}
        del bm, sb
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ drop-in surface
def e2e_dropin(args, prot, batch, dev, steps):
    """The same configs[1] pass driven EXACTLY as INTEGRATION.md section 1 / test.py:495-582 drives it, one ensemble member batch at a
    time being the reference's own loop structure replaced by a 10-row batch: factory model, create_diffusion, p_sample_loop(model.forward),
    get_norm_feature, latent_decode, ic_to_xyz -- host batch dict in, host coordinates out."""
    from codlad_b200 import weights
    from codlad_b200.diffusion import create_diffusion
    from codlad_b200.latent_model import MPNN_models
    from codlad_b200.utils_ic import ic_to_xyz
    from codlad_b200.vae_model import VAE, get_norm_feature
    from codlad_b200 import synthetic
    model = MPNN_models["mpnn_diffusion"](input_size=3, unconditional=True, diffusion="diffusion", precision=args.precision)
    model.load_state_dict(weights.init_denoiser_state(0))
    vae = VAE("N6")
    vae.load_state_dict(weights.init_vae_decode_state(0))
    diffusion = create_diffusion(str(T_STEPS))
    mb = synthetic.collate(prot, frames=[0] * ENSEMBLE)             # the ensemble as a batch of 10 copies of the frame (reference schema)
    mb = {k: v.to(dev) if torch.is_tensor(v) else v for k, v in mb.items()}          # test.py:487 batch_to(batch, device)
    mask = torch.ones(ENSEMBLE, L_RES, dtype=torch.bool, device=dev)
    og = mb["OG_CG_nxyz"].reshape(-1, L_RES + 2, 4)

    def one_pass():
        z = torch.randn(ENSEMBLE, L_RES, 3, device=dev)
        samples = diffusion.p_sample_loop(model.forward, z.shape, z, clip_denoised=False, model_kwargs=dict(y=None, mask=mask, batch=mb), device=dev)
        samples = get_norm_feature(samples, "N6", norm_channel=True, norm_single=False, norm_in=False, dataname="PED")
        _, ic_recon = vae.latent_decode(samples, mask, mb)
        xyz = ic_to_xyz(og, ic_recon.reshape(-1, L_RES, 13, 3), prot.info)
        return xyz.cpu()

    for _ in range(2):
        one_pass()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_pass()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    return {"value": L_RES * ENSEMBLE / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "path": "MPNN_models factory + create_diffusion.p_sample_loop(model.forward) + get_norm_feature + VAE.latent_decode + ic_to_xyz (un-doubled 10-row batch)",
            "scope": "ONE GPU (rank 0 alone), whatever --gpus is: compare with e2e / n_gpus"}


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="codlad_b200", choices=["codlad_b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("CB2_PRECISION", "f16"), choices=["f16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + ["metrics", "c5"],
                    help="c2 = the bench line; c3 / c4 = per-GPU shards of the larger configs; c5 = the train_latent step; metrics = the evaluation-step kernel")
    ap.add_argument("--train-gemm", default="tf32", choices=["tf32", "fp32"], help="c5: TF32 tensor-core GEMMs (the reference's arithmetic) or fp32 SIMT")
    ap.add_argument("--micro-batch", type=int, default=64, help="c5: proteins per forward/backward (gradients accumulate to the per-rank batch)")
    ap.add_argument("--scale", default="all", choices=["all", "c3", "c4", "none"], help="scale_checks jobs run through the sharded driver")
    ap.add_argument("--scale-passes", type=int, default=2)
    ap.add_argument("--lean", action="store_true", help="only value / e2e / roofline (no roofline_all, scale_checks, drop-in, CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of rank 0's last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("metrics", "c5")):
        ap.error("--dump-outputs writes the outputs of the sampling path: --impl codlad_b200 with --workload c2, c3 or c4")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload in ("metrics", "c5"):
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: codlad_b200 has no CPU fallback")
        return run_metrics(args) if args.workload == "metrics" else run_train(args)
    args.warmup = max(args.warmup, 3)

    from codlad_b200 import distributed as D
    rank, world, local = D.env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: codlad_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    D.init_from_env("nccl", local)
    torch.set_grad_enabled(False)
    from codlad_b200 import sampler, weights

    dev = torch.device("cuda", local)
    wl = WORKLOADS[args.workload]
    prot, batch, fs = _workload(rank, args.workload, world)
    fs.pin()
    angle = wl["vae"] in ("K3", "K4")
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0, angle, (wl["vae"], sampler.VAE_DATA[wl["vae"]])),
                            wl["vae"], k_neighbors=wl["k"], num_sampling_steps=T_STEPS, precision=args.precision)
    plan = bm.upload(fs)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    # ---- device-resident throughput: inputs already in HBM, per-step CUDA events, L2 flushed between steps
    for _ in range(args.warmup):
        bm.sample(plan, fs, generator=gen)
    D.barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = plan.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in ev:
        out = None                      # free the previous step's outputs before this step allocates, as if they were not kept
        flush.fill_(1)
        a.record()
        out = bm.sample(plan, fs, generator=gen)
        b.record()
    D.barrier()
    launches = plan.launches - l0
    ms_dev = D.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) / args.steps, dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)           # before the passes below overwrite the plan's buffers
    del out
    residues = fs.NB * fs.L * world
    value = residues / (ms_dev * 1e-3)

    # ---- end to end through the host API: pinned host inputs -> H2D -> whole path -> D2H coordinates
    h2d = fs.host_bytes()
    for _ in range(2):
        xyz = bm.backmap_host(fs, generator=gen)
    d2h = xyz.numel() * xyz.element_size()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        bm.backmap_host(fs, generator=gen)
    torch.cuda.synchronize()
    ms_e2e = D.max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps, dev)
    D.barrier()
    clk = clocks.stop() if clocks else None

    # ---- dominant kernel alone: encoder edge-update MLP (3 chained 128x128 GEMMs per edge + LN/adaLN epilogue)
    roof = roof_all = None
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get(f"{args.workload}_{args.precision}", {})
    if rank == 0:
        peaks = _peaks()
        mode = 1
        edges = fs.NB * fs.L * plan.K
        ms_k, ms_warm = (v * 1e-3 for v in _time_stage(lambda: plan.run_edge_kernel(mode, 1), flush, reps=20))
        achieved = EDGE_FLOPS[mode] * edges / (ms_k * 1e-3) / 1e12
        # `traffic`: dram bytes of THIS launch (same workload, same layer, same precision) from the committed ncu --set full capture
        # (profiles/traffic.json, written by tools/ncu_traffic.py); null when no capture of this workload exists
        roof = {"kernel": f"edge kernel mode {mode} (encoder edge update, layer 1), {args.precision} tier", "bound": "tensor",
                "achieved": achieved, "peak": peaks["tflops_burst"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops_burst"],
                "traffic": traffic.get("edge update, encoder (edge kernel mode 1)"),
                "peak_source": peaks["source"] + ", burst (kernel timed alone)", "us_per_launch": ms_k * 1e3,
                "us_per_launch_l2_resident": ms_warm * 1e3, "achieved_l2_resident": EDGE_FLOPS[mode] * edges / (ms_warm * 1e-3) / 1e12,
                "frac_l2_resident": EDGE_FLOPS[mode] * edges / (ms_warm * 1e-3) / 1e12 / peaks["tflops_burst"],
                "flops_per_launch": EDGE_FLOPS[mode] * edges, "algorithmic_bytes_per_launch": edges * 128 * 2 * (2 if args.precision == "f16" else 4)}
        if not args.lean:
            roof_all = roofline_all(plan, bm, fs, flush, peaks, args.precision, traffic)

    dropin = None
    if rank == 0 and not args.lean and args.workload == "c2":
        dropin = e2e_dropin(args, prot, batch, dev, args.steps)
    del plan, bm
    torch.cuda.empty_cache()
    scale = None
    if not args.lean and args.scale != "none":
        scale = scale_checks(args, D, dev, rank, world)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.lean and args.workload == "c2":
        cpu = cpu_port_sample(denoiser_steps=2)
        cpu["anchor_configs0"] = cpu_anchor_c1()

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (tcgen05, fp32 accumulate)" if args.precision == "f16" else "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "residues_per_step_per_gpu": fs.NB * fs.L, "diffusion_steps": T_STEPS, "k_neighbors": wl["k"],
                       "weights": "random init (seed 0), adaLN layers re-randomised", "l2": "flushed between timed steps (512 MiB fill)",
                       "sharding": f"{fs.F} frame(s) x {fs.NB // fs.F} member(s) per GPU, no collective"},
            "e2e": {"value": residues / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e},
            "e2e_dropin": dropin, "gpu_launches": launches, "clocks": clk, "roofline": roof, "roofline_all": roof_all,
            "scale_checks": scale, "cpu_baseline": cpu,
        }))
    D.shutdown()


if __name__ == "__main__":
    main()
