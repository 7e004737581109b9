"""Partial-noise refinement and warm-started trajectory backmapping at configs[1] (one 300-residue frame x 10 members, N6 decoder,
f16 tier).  Prints one JSON line with:

  * device time of one backmapping pass (sampling loop + decode): Backmapper.refine at several starts against Backmapper.sample,
    for DDPM-100 and DDIM-25 (eta = 0), variants alternating in every round, one plan per variant so that no timed pass
    re-captures its graph;
  * a 32-frame synthetic trajectory (synthetic.trajectory) x 10 members, host wall time with host inputs in and host coordinates
    out: 32 independent backmap_host calls against backmap_trajectory at DDPM-100 / 25 steps and DDIM-25 / 6 steps, chunks 1 and
    4; frames/s, residues/s, and the share of wall time the host spends converting and uploading frame sets (from a replica of
    backmap_trajectory's loop with that part timed);
  * the mean residue_motion between consecutive frames of both, which with random-init weights shows the mechanics of the warm
    start only, not the quality of a trained model.

    python tools/bench_refine.py [--rounds 3] [--passes 10] [--warmup 3]

Each timed device pass is bracketed by CUDA events with the L2 overwritten (512 MiB fill) before it, as bench.py does.  The card's
name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# name, sampler, T, refinement starts timed, start of the trajectory runs
SAMPLERS = [("ddpm100", "ddpm", 100, [10, 25, 50, 100], 25), ("ddim25", "ddim", 25, [6, 12, 25], 6)]
FRAMES = 32
CHUNKS = [1, 4]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="rounds; every round times every variant (at least 3)")
    ap.add_argument("--passes", type=int, default=10, help="timed device passes of one variant per round")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_refine.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from bench_inpaint import gpu_info
    from codlad_b200 import batching, sampler, synthetic, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    wl = bench.WORKLOADS["c2"]
    _, _, fs = bench._workload(0, "c2")
    fs.pin()
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    make = lambda kind, T: sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=T, precision="f16",
                                              sampler=kind)

    # ---- device time per pass ----------------------------------------------------------------------------------------------------
    bms, plans, latents = {}, {}, {}
    for name, kind, T, starts, _ in SAMPLERS:
        for s in [0] + starts:                                   # 0 = plain sample()
            bm = make(kind, T)
            bms[(name, s)], plans[(name, s)] = bm, bm.upload(fs)
        latents[name] = bms[(name, 0)].sample(plans[(name, 0)], fs, generator=gen)["latent"].clone()

    def run(name, s):
        bm, plan = bms[(name, s)], plans[(name, s)]
        if s == 0:
            return bm.sample(plan, fs, generator=gen)
        return bm.refine(plan, fs, latents[name], s, generator=gen)

    variants = list(bms)
    for v in variants:
        for _ in range(args.warmup):
            run(*v)
    torch.cuda.synchronize()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    times = {v: [] for v in variants}
    launches = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:                                     # variants alternate inside every round
            plan = plans[v]
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.passes)]
            l0 = plan.launches
            for a, b in ev:
                flush.fill_(1)
                a.record()
                run(*v)
                b.record()
            torch.cuda.synchronize()
            times[v] += [a.elapsed_time(b) for a, b in ev]
            launches[v].append((plan.launches - l0) / args.passes)
    residues = fs.NB * fs.L
    passes = {}
    for name, kind, T, starts, _ in SAMPLERS:
        plain = statistics.median(times[(name, 0)])
        for s in [0] + starts:
            t = times[(name, s)]
            med = statistics.median(t)
            passes[f"{name}_plain" if s == 0 else f"{name}_refine{s}"] = {
                "sampler": kind, "T": T, "steps_run": T if s == 0 else s, "call": "sample" if s == 0 else "refine",
                "ms_per_pass_median": med, "ms_per_pass_min": min(t), "ms_per_pass_max": max(t),
                "residues_per_s": residues / (med * 1e-3), "over_plain_time": med / plain,
                "launches_per_pass": statistics.median(launches[(name, s)])}
    del bms, plans
    torch.cuda.empty_cache()

    # ---- 32-frame trajectory, host in / host out -----------------------------------------------------------------------------------
    prot = synthetic.trajectory(wl["L"], FRAMES, seed=1002)
    batches = [synthetic.collate(prot, [f]) for f in range(FRAMES)]
    E = wl["ensemble"]
    frame_fs = sampler.frames_from_batch(batches[0], prot.info, E)

    def independent(bm):
        out = []
        for batch in batches:
            f_fs = sampler.frames_from_batch(batch, prot.info, E).pin()
            out.append(bm.backmap_host(f_fs, generator=gen).clone().view(E, -1, 3))
        return torch.stack(out)

    def host_share(bm, steps, chunks):
        """backmap_trajectory's loop with the host conversion + upload of every pass timed: (that time, total wall) in ms."""
        runs = sampler.trajectory_chunks(FRAMES, chunks)
        torch.cuda.synchronize()
        t0, host = time.perf_counter(), 0.0
        res = None
        for p in range(runs[0][1]):
            h0 = time.perf_counter()
            frames = [s + min(p, n - 1) for s, n in runs]
            p_fs = sampler.frames_from_batch(batching.merge_batches([batches[f] for f in frames]), prot.info, E)
            plan = bm.upload(p_fs)
            torch.cuda.synchronize()
            host += time.perf_counter() - h0
            res = bm.sample(plan, p_fs, generator=gen) if p == 0 else bm.refine(plan, p_fs, res["latent"], steps, generator=gen)
            res["xyz"].cpu()
        torch.cuda.synchronize()
        return host * 1e3, (time.perf_counter() - t0) * 1e3

    def motion(bm, xyz):
        """mean residue_motion between consecutive frames of host xyz [FRAMES, E, Na, 3]"""
        m = [bm.residue_motion(frame_fs, xyz[f].reshape(-1, 3).to(dev), xyz[f + 1].reshape(-1, 3).to(dev)) for f in range(FRAMES - 1)]
        m = torch.stack(m)
        return float(m[~torch.isnan(m)].mean())

    traj = {}
    for name, kind, T, _, steps in SAMPLERS:
        bm_ind, bm_traj = make(kind, T), make(kind, T)
        jobs = [("independent", None)] + [(f"trajectory_chunks{c}", c) for c in CHUNKS]
        fn = {"independent": lambda: independent(bm_ind)}
        for label, c in jobs[1:]:
            fn[label] = (lambda c=c: bm_traj.backmap_trajectory(batches, prot.info, num_ensemble=E, steps=steps, chunks=c, generator=gen))
        for label, _ in jobs:                                  # warm-up: graphs, plans, pinned buffers
            fn[label]()
        wall = {label: [] for label, _ in jobs}
        share = {label: [] for label, c in jobs if c is not None}
        outs = {}
        for _ in range(args.rounds):
            for label, c in jobs:                              # alternating
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                outs[label] = fn[label]()
                wall[label].append((time.perf_counter() - t0) * 1e3)
                if c is not None:
                    h, w = host_share(bm_traj, steps, c)
                    share[label].append(h / w)
        for label, c in jobs:
            med = statistics.median(wall[label])
            traj[f"{name}_{label}"] = {
                "sampler": kind, "T": T, "refine_steps": None if c is None else steps, "chunks": c,
                "wall_ms_median": med, "wall_ms_min": min(wall[label]), "wall_ms_max": max(wall[label]),
                "frames_per_s": FRAMES / (med * 1e-3), "residues_per_s": FRAMES * E * wl["L"] / (med * 1e-3),
                "host_convert_upload_share_median": statistics.median(share[label]) if c is not None else None,
                "mean_residue_motion_consecutive_frames_A": motion(bm_traj, outs[label])}
        for label, c in jobs[1:]:
            traj[f"{name}_{label}"]["speedup_over_independent"] = \
                traj[f"{name}_independent"]["wall_ms_median"] / traj[f"{name}_{label}"]["wall_ms_median"]

    print(json.dumps({
        "metric": "partial-noise refinement (Backmapper.refine) and warm-started trajectory backmapping (backmap_trajectory)",
        "gpu": gpu_info(), "workload": "configs[1]: PED-like 300-residue IDP, N6, num_ensemble=10",
        "precision": "f16 (tcgen05, fp32 accumulate)", "weights": "random init (seed 0)",
        "device_passes": {"unit": "ms per pass (sampling loop + decode), CUDA events", "l2": "flushed before every timed pass (512 MiB fill)",
                          "rounds": args.rounds, "passes_per_round": args.passes, "variants": passes},
        "trajectory": {"unit": "host wall time per 32-frame trajectory, host inputs in, host coordinates out",
                       "frames": FRAMES, "members": E, "residues": wl["L"], "ca_step_rms_A": 0.05, "rounds": args.rounds,
                       "host_share": "frames_from_batch + upload (synchronised) over wall time, in a replica of backmap_trajectory's loop",
                       "motion_note": "random-init weights: residue_motion shows the mechanics of the warm start, not sample quality",
                       "variants": traj},
    }, default=lambda v: None if isinstance(v, float) and math.isnan(v) else v))


if __name__ == "__main__":
    main()
