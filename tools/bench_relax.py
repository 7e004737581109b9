"""Restrained clash relaxation, measured: (1) one cb2_plan_relax call at the default iterations (Backmapper.relax's kernel work,
Plan.relax) on decoded samples of configs[1] (one 300-residue frame x 10 members, N6) and configs[3] (one 2000-residue frame x 32
members, K4, k_neighbors 48), with clash pairs under 1.2 A before and after; (2) at configs[1], a DDPM-100 and a DDIM-25 pass
(Backmapper.sample) for scale, alternated with the relax calls in one process; (3) trajectory frames/s of backmap_coords at DDIM-25 /
6 steps with and without relax=.  Prints one JSON line.

    python tools/bench_relax.py [--rounds 5] [--calls 20] [--warmup 3] [--frames 32]

Every timed call or pass is bracketed by CUDA events with the L2 overwritten (512 MiB fill) before it, as bench.py does.  The
structures come from random-init weights, so their clash counts show the mechanics only, not model quality.  The card's name and
power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.bench_inpaint import gpu_info  # noqa: E402
from tools.bench_repair import summary, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5, help="rounds; every round times every variant (at least 3)")
    ap.add_argument("--calls", type=int, default=20, help="timed calls or passes of one variant per round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=32, help="trajectory frames (L = 300, 10 members)")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_relax.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from codlad_b200 import sampler, synthetic, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    dsd = weights.init_denoiser_state(0)
    it = sampler.RELAX_ITERATIONS

    variants, cases = {}, {}
    for cfg in ("c2", "c4"):
        wl = bench.WORKLOADS[cfg]
        _, _, fs = bench._workload(0, cfg)
        vsd = weights.init_vae_decode_state(0, angle_variant=wl["vae"] in ("K3", "K4"))
        bm = sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=10, precision="f16")
        plan = bm.upload(fs)
        out = {k: v.clone() for k, v in bm.sample(plan, fs, generator=gen).items()}
        res = bm.relax(plan, fs, out)
        l0 = plan.launches
        plan.relax(out["xyz"], 1.2, it)
        cases[cfg] = {"residues": fs.NB * fs.L, "atoms": fs.total_atoms, "iterations": it, "launches_per_call": plan.launches - l0,
                      "clash_pairs_1.2_before": res["clash_pairs"][0].tolist(), "clash_pairs_1.2_after": res["clash_pairs"][1].tolist(),
                      "max_shift_A": max(res["max_shift"].tolist()), "max_restraint_dev_A": max(res["max_restraint_dev"].tolist())}
        variants[f"relax_{cfg}"] = (lambda plan=plan, xyz=out["xyz"]: plan.relax(xyz, 1.2, it))
    wl = bench.WORKLOADS["c2"]
    _, _, fs = bench._workload(0, "c2")
    vsd = weights.init_vae_decode_state(0)
    for name, kind, steps in (("ddpm100", "ddpm", 100), ("ddim25", "ddim", 25)):
        bm = sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=steps, precision="f16", sampler=kind)
        plan = bm.upload(fs)
        variants[f"pass_{name}_c2"] = (lambda bm=bm, plan=plan: bm.sample(plan, fs, generator=gen))
    for fn in variants.values():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(args.rounds):
        for k, fn in variants.items():                   # variants alternate inside every round
            times[k] += timed(fn, args.calls, flush)
    stats = {k: summary(t) for k, t in times.items()}
    ratio = stats["relax_c2"]["ms_median"] / stats["pass_ddim25_c2"]["ms_median"]

    # trajectory frames/s, DDIM-25 / 6 refinement steps, with and without relax
    bm = sampler.Backmapper(dsd, vsd, "N6", num_sampling_steps="ddim25", precision="f16", sampler="ddim")
    prot = synthetic.trajectory(300, args.frames, seed=42)
    traj = {}
    for opt in (None, {}, None, {}):                     # alternated; the second of each is kept
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bm.backmap_coords(prot.ca_full, prot.restype_full, prot.info, num_ensemble=10, steps=6, chunks=8, seed=1, relax=opt)
        torch.cuda.synchronize()
        traj["relax" if opt is not None else "plain"] = args.frames / (time.perf_counter() - t0)
    print(json.dumps({
        "metric": "one cb2_plan_relax call at default iterations vs sampling passes; trajectory frames/s with and without relax",
        "unit": "ms", "gpu": gpu_info(), "precision": "f16 decode (tcgen05, fp32 accumulate); relax is fp32",
        "weights": "random init (seed 0)", "l2": "flushed before every timed call or pass (512 MiB fill)",
        "cases": {"configs[1] (c2: 300 x 10, N6)": cases["c2"], "configs[3] (c4: 2000 x 32, K4, K 48)": cases["c4"]},
        "timings": stats, "relax_c2_over_ddim25_pass": ratio, "target_under_10pct_of_ddim25_met": ratio < 0.10,
        "trajectory_frames_per_s": {"workload": f"{args.frames} frames x 10 members, L 300, DDIM-25 / 6 steps, chunks 8", **traj},
        "rounds": args.rounds, "calls_per_round": args.calls,
    }))


if __name__ == "__main__":
    main()
