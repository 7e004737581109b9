"""Sharded trajectory backmapping (ShardedBackmapper.backmap_coords) on N GPUs.  Run once per world size, N = 1 first:

    torchrun --nproc_per_node N tools/bench_traj_sharded.py [--rounds 3] [--ref-dir DIR]

Workloads (f16 tier, N6 decoder, random-init weights, DDIM-25 with 6 refinement steps per frame, 10 members, seeded keyed noise):

  * traj256: one 256-frame synthetic.trajectory at L = 300, chunks 8;
  * atlas_c1 / atlas_c4: an ATLAS-like job of 32 trajectories x 32 frames, L drawn from U[200, 500] with a fixed seed, chunks 1
    and 4.

For each: frames/s and residues/s (frames x L x members), the compute time of every rank (CUDA events around its local units, max
over ranks) and the wall time of the call on a synchronised host clock, gather on rank 0 included (max over ranks); the load
imbalance (max / mean) of the partition's cost model and of the measured compute times; and whether rank 0's output equals the
N = 1 output, which the N = 1 run stores in --ref-dir (a temporary directory, outside the tree), with the largest difference when
it does not.  Medians over --rounds timed calls after one untimed call.  Rank 0 prints one JSON line with the card's name and power
limit."""
import argparse
import json
import os
import random
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

T, STEPS, ENSEMBLE, SEED = 25, 6, 10, 0x7A5C_5EED


def workloads():
    from codlad_b200 import synthetic
    traj = synthetic.trajectory(300, 256, seed=9001)
    rnd = random.Random(2024)
    atlas = [synthetic.trajectory(rnd.randint(200, 500), 32, seed=9100 + i) for i in range(32)]
    job = lambda prots: [(p.ca_full, p.restype_full, p.info) for p in prots]
    return {"traj256": (job([traj]), 8), "atlas_c1": (job(atlas), 1), "atlas_c4": (job(atlas), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="timed calls per workload (at least 3)")
    ap.add_argument("--ref-dir", default=os.path.join(tempfile.gettempdir(), "codlad_bench_traj_sharded"),
                    help="where the N = 1 run stores its outputs and larger N compare against them")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_traj_sharded.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import torch.distributed as dist
    from bench_inpaint import gpu_info
    from codlad_b200 import distributed, sampler, weights

    rank, world, local = distributed.env_rank_world()
    torch.cuda.set_device(local)
    distributed.init_from_env("nccl", local)
    torch.set_grad_enabled(False)
    bm = sampler.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", k_neighbors=64,
                            num_sampling_steps=T, precision="f16", sampler="ddim")
    sb = sampler.ShardedBackmapper(bm, rank, world)

    def per_rank(value):
        """value of every rank, as a list."""
        if world == 1:
            return [float(value)]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = float(value)
        dist.all_reduce(t)
        return t.tolist()

    results = {}
    for name, (job, chunks) in workloads().items():
        n_frames = [ca.shape[0] for ca, _, _ in job]
        lengths = [ca.shape[1] - 2 for ca, _, _ in job]
        runs, parts = sampler.partition_trajectory_units(n_frames, lengths, ENSEMBLE, STEPS, T, chunks, world, bm.k_neighbors)
        cost = lambda t, c: lengths[t] * min(bm.k_neighbors, lengths[t]) * ENSEMBLE * (T + (runs[t][c][1] - 1) * STEPS)
        loads = [sum(cost(t, c) for t, c in p) for p in parts]
        timing = {}

        def compute(*a, **k):
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            res = sb.backmap_coords_local(*a, **k)
            end.record()
            end.synchronize()
            timing["compute_ms"] = start.elapsed_time(end)
            return res

        def call():
            timing["compute_ms"] = 0.0                     # a rank with no unit computes nothing
            distributed.barrier()
            t0 = time.perf_counter()
            out = sb.backmap_coords(job, num_ensemble=ENSEMBLE, steps=STEPS, chunks=chunks, seed=SEED, _compute=compute)
            wall = (time.perf_counter() - t0) * 1e3
            return out, per_rank(timing["compute_ms"]), max(per_rank(wall))

        out, _, _ = call()                                  # warm-up: plans, graphs, the lazy module loads
        compute_ms, wall_ms = [], []
        imbalance = []
        for _ in range(args.rounds):
            out, comp, wall = call()
            compute_ms.append(max(comp))
            wall_ms.append(wall)
            imbalance.append(max(comp) / (sum(comp) / world))
        frames = sum(n_frames)
        residues = sum(n * L for n, L in zip(n_frames, lengths)) * ENSEMBLE
        comp_med, wall_med = statistics.median(compute_ms), statistics.median(wall_ms)
        entry = {
            "trajectories": len(job), "frames": frames, "L": lengths[0] if len(job) == 1 else [min(lengths), max(lengths)],
            "chunks": chunks, "units": sum(len(r) for r in runs), "units_per_rank": [len(p) for p in parts],
            "compute_ms_max_over_ranks_median": comp_med, "compute_ms_min": min(compute_ms), "compute_ms_max": max(compute_ms),
            "wall_ms_median": wall_med, "wall_ms_min": min(wall_ms), "wall_ms_max": max(wall_ms),
            "frames_per_s_compute": frames / (comp_med * 1e-3), "frames_per_s_wall": frames / (wall_med * 1e-3),
            "residues_per_s_compute": residues / (comp_med * 1e-3), "residues_per_s_wall": residues / (wall_med * 1e-3),
            "imbalance_cost_model": max(loads) / (sum(loads) / world), "imbalance_measured_median": statistics.median(imbalance),
        }
        if rank == 0:
            ref_path = os.path.join(args.ref_dir, f"{name}.pt")
            if world == 1:
                os.makedirs(args.ref_dir, exist_ok=True)
                torch.save(out, ref_path)
                entry["equals_n1"] = "reference (this run)"
            elif os.path.exists(ref_path):
                ref = torch.load(ref_path)
                same = all(torch.equal(a, b) for a, b in zip(out, ref))
                entry["equals_n1"] = same
                entry["frames_bit_identical"] = sum(int(torch.equal(a[f], b[f])) for a, b in zip(out, ref) for f in range(a.shape[0]))
                if not same:
                    entry["max_abs_diff"] = max(float((a - b).abs().max()) for a, b in zip(out, ref))
                    entry["max_rel_err"] = max(float((a - b).norm() / b.norm()) for a, b in zip(out, ref))
            else:
                entry["equals_n1"] = "not compared: no N = 1 output in --ref-dir"
        results[name] = entry
        del out

    if rank == 0:
        print(json.dumps({
            "metric": "sharded trajectory backmapping (ShardedBackmapper.backmap_coords)", "gpu": gpu_info(), "world": world,
            "gpus_visible": torch.cuda.device_count(), "precision": "f16 (tcgen05, fp32 accumulate)", "weights": "random init (seed 0)",
            "sampler": f"DDIM-{T}, eta 0, {STEPS} refinement steps per frame", "members": ENSEMBLE, "rounds": args.rounds,
            "units": {"compute": "CUDA events around a rank's local units (host work inside included), max over ranks",
                      "wall": "synchronised host clock from a barrier to the call's return, gather on rank 0 included, max over ranks",
                      "residues": "frames x L x members"},
            "workloads": results}))
    distributed.shutdown()


if __name__ == "__main__":
    main()
