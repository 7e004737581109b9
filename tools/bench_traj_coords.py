"""Trajectory backmapping from a coordinate array (Backmapper.backmap_coords, geometry built on the device) against batch dicts
(Backmapper.backmap_trajectory, frames_from_batch + upload every pass).  Prints one JSON line with:

  * the 32-frame x 10-member synthetic.trajectory at L = 300 (configs[1]'s size, N6 decoder, f16 tier) through both methods at
    DDPM-100 / 25 refinement steps and DDIM-25 / 6 steps, chunks 1 and 4, host coordinates in and host coordinates out: frames/s,
    the share of wall time the per-pass geometry step takes (from a replica of the pass loop with that step synchronised and
    timed: frames_from_batch + upload for batch dicts, update_coords for the coordinate array), and whether the outputs of the two
    methods are identical;
  * one geometry update alone: update_coords against frames_from_batch + upload of the same frames, at 1 frame x 10 members and 4
    frames x 10 members;
  * the radius-graph kernels (cb2_radius_graph_rows + _fill) at L = 300 and L = 2000, CUDA events over many launches.

    python tools/bench_traj_coords.py [--rounds 3]

Variants alternate inside every round.  The card's name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

# name, sampler, T, refinement steps per frame
SAMPLERS = [("ddpm100", "ddpm", 100, 25), ("ddim25", "ddim", 25, 6)]
FRAMES, L, ENSEMBLE = 32, 300, 10
CHUNKS = [1, 4]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="rounds; every round times every variant (at least 3)")
    ap.add_argument("--updates", type=int, default=20, help="timed geometry updates of one variant per round")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_traj_coords.py needs a CUDA device: codlad_b200 has no CPU fallback")
    from bench_inpaint import gpu_info
    from codlad_b200 import _native as N
    from codlad_b200 import batching, engine, sampler, synthetic, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    make = lambda kind, T: sampler.Backmapper(dsd, vsd, "N6", k_neighbors=64, num_sampling_steps=T, precision="f16", sampler=kind)
    prot = synthetic.trajectory(L, FRAMES, seed=1002)
    batches = [synthetic.collate(prot, [f]) for f in range(FRAMES)]
    sync = torch.cuda.synchronize

    # ---- the trajectory both ways ----------------------------------------------------------------------------------------------------
    def geometry_share(bm, steps, chunks, coords):
        """The pass loop of the trajectory methods with the geometry step of every pass synchronised and timed: (that time, wall) ms."""
        runs = sampler.trajectory_chunks(FRAMES, chunks)
        t = {"geo": 0.0}
        if coords:
            fs = sampler.frames_from_coords(prot.ca_full[[s for s, _ in runs]], prot.restype_full, prot.info, ENSEMBLE)
            ca = {}

        def frame_set(p, frames):
            sync()
            t0 = time.perf_counter()
            if coords:
                plan = bm.upload(fs) if p == 0 else bm.plan_for(fs)
                if p == 0:
                    ca["all"] = prot.ca_full.to(dev)
                bm.update_coords(plan, fs, ca["all"][frames])
                out = plan, fs
            else:
                p_fs = sampler.frames_from_batch(batching.merge_batches([batches[f] for f in frames]), prot.info, ENSEMBLE)
                out = bm.upload(p_fs), p_fs
            sync()
            t["geo"] += time.perf_counter() - t0
            return out

        sync()
        t0 = time.perf_counter()
        bm._trajectory_passes(FRAMES, ENSEMBLE, steps, runs, frame_set, gen)
        return t["geo"] * 1e3, (time.perf_counter() - t0) * 1e3

    gen = torch.Generator(device=dev).manual_seed(1234)
    traj = {}
    for name, kind, T, steps in SAMPLERS:
        bm_b, bm_c = make(kind, T), make(kind, T)
        jobs = [(f"{m}_chunks{c}", m, c) for c in CHUNKS for m in ("batches", "coords")]

        def run(method, c, seed=None):
            g = gen if seed is None else torch.Generator(device=dev).manual_seed(seed)
            if method == "batches":
                return bm_b.backmap_trajectory(batches, prot.info, num_ensemble=ENSEMBLE, steps=steps, chunks=c, generator=g)
            return bm_c.backmap_coords(prot.ca_full, prot.restype_full, prot.info, num_ensemble=ENSEMBLE, steps=steps, chunks=c,
                                       generator=g)

        same = {c: bool(torch.equal(run("batches", c, 77), run("coords", c, 77))) for c in CHUNKS}     # also the warm-up
        wall = {j: [] for j, _, _ in jobs}
        share = {j: [] for j, _, _ in jobs}
        for _ in range(args.rounds):
            for label, method, c in jobs:
                sync()
                t0 = time.perf_counter()
                run(method, c)
                wall[label].append((time.perf_counter() - t0) * 1e3)
                g, w = geometry_share(bm_c if method == "coords" else bm_b, steps, c, method == "coords")
                share[label].append(g / w)
        for label, method, c in jobs:
            med = statistics.median(wall[label])
            traj[f"{name}_{label}"] = {
                "sampler": kind, "T": T, "refine_steps": steps, "chunks": c, "method": method,
                "call": "backmap_trajectory" if method == "batches" else "backmap_coords",
                "wall_ms_median": med, "wall_ms_min": min(wall[label]), "wall_ms_max": max(wall[label]),
                "frames_per_s": FRAMES / (med * 1e-3), "geometry_share_median": statistics.median(share[label]),
                "outputs_identical_to_batches": same[c]}
        for c in CHUNKS:
            b, k = traj[f"{name}_batches_chunks{c}"], traj[f"{name}_coords_chunks{c}"]
            k["speedup_over_batches"] = b["wall_ms_median"] / k["wall_ms_median"]
        del bm_b, bm_c

    # ---- one geometry update ---------------------------------------------------------------------------------------------------------
    bm = make("ddim", 25)
    update = {}
    for F in (1, 4):
        frames = list(range(F))
        fs0 = sampler.frames_from_batch(batching.merge_batches([batches[f] for f in frames]), prot.info, ENSEMBLE)
        plan = bm.upload(fs0)
        ca = prot.ca_full.to(dev)
        sets = [[(f + k) % FRAMES for f in frames] for k in range(FRAMES)]

        def host_path(k):
            fs = sampler.frames_from_batch(batching.merge_batches([batches[f] for f in sets[k]]), prot.info, ENSEMBLE)
            bm.upload(fs)

        def device_path(k):
            bm.update_coords(plan, fs0, ca[sets[k]])

        times = {"frames_from_batch_upload": [], "update_coords": []}
        for fn in (host_path, device_path):
            fn(1)
        for _ in range(args.rounds):
            for label, fn in (("frames_from_batch_upload", host_path), ("update_coords", device_path)):
                for k in range(args.updates):
                    sync()
                    t0 = time.perf_counter()
                    fn(k % FRAMES)
                    sync()
                    times[label].append((time.perf_counter() - t0) * 1e3)
        update[f"F{F}_NB{F * ENSEMBLE}"] = {
            label: {"ms_median": statistics.median(t), "ms_min": min(t), "ms_max": max(t)} for label, t in times.items()}
        update[f"F{F}_NB{F * ENSEMBLE}"]["speedup"] = (update[f"F{F}_NB{F * ENSEMBLE}"]["frames_from_batch_upload"]["ms_median"] /
                                                      update[f"F{F}_NB{F * ENSEMBLE}"]["update_coords"]["ms_median"])

    # ---- radius-graph kernels ----------------------------------------------------------------------------------------------------------
    kernels = {}
    for n in (300, 2000):
        p = synthetic.make_protein(n, 1, seed=n)
        X = p.ca_full[:, 1:-1].contiguous().to(dev)
        lengths = torch.full((1,), n, dtype=torch.int32, device=dev)
        row, col = engine.radius_graph(X, lengths)
        reps = 200
        res = []
        for _ in range(args.rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                N.check(N.lib().cb2_radius_graph_rows(N.dptr(X), N.dptr(lengths), 1, n, 21.0, N.dptr(row), N.stream_ptr()), "rows")
                N.check(N.lib().cb2_radius_graph_fill(N.dptr(X), N.dptr(lengths), 1, n, 21.0, N.dptr(row), N.dptr(col), N.stream_ptr()),
                        "fill")
            b.record()
            sync()
            res.append(a.elapsed_time(b) / reps)
        kernels[f"L{n}"] = {"us_rows_plus_fill_median": 1e3 * statistics.median(res), "us_min": 1e3 * min(res), "edges": int(col.numel()),
                            "launches": 3}

    print(json.dumps({
        "metric": "trajectory backmapping from a coordinate array (backmap_coords) against batch dicts (backmap_trajectory)",
        "gpu": gpu_info(), "workload": f"synthetic.trajectory: {FRAMES} frames x {ENSEMBLE} members, L = {L}, N6, 0.05 A RMS step",
        "precision": "f16 (tcgen05, fp32 accumulate)", "weights": "random init (seed 0)", "rounds": args.rounds,
        "trajectory": {"unit": "host wall time per trajectory, host coordinates in, host coordinates out",
                       "geometry_share": "per-pass geometry step (synchronised) over wall time, in a replica of the pass loop",
                       "variants": traj},
        "geometry_update": {"unit": "ms per update, synchronised host clock", "updates_per_round": args.updates, "variants": update},
        "radius_graph_kernels": {"unit": "us per graph (count + scan + fill), CUDA events over 200 graphs", "variants": kernels},
    }))


if __name__ == "__main__":
    main()
