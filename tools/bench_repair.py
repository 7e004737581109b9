"""Clash-driven repair, measured: (1) the per-residue clash launches of cb2_plan_residue_clashes (residue bounds, clash counts,
keep mask; one call) on decoded samples of configs[1] (one 300-residue frame x 10 members, N6) and configs[3] (one 2000-residue
frame x 32 members, K4, k_neighbors 48); (2) at configs[1], one repair round (Backmapper.repair with max_rounds=1) against a plain
pass (Backmapper.sample), for DDPM-100 and DDIM-25 (eta = 0), alternated in one process.  Prints one JSON line.

    python tools/bench_repair.py [--rounds 5] [--passes 10] [--warmup 3] [--calls 50]

Every timed call or pass is bracketed by CUDA events with the L2 overwritten (512 MiB fill) before it, as bench.py does.  The
structures come from random-init weights, so their clash counts say nothing about real models; the threshold of the repair
round is the reference's 1.2 A unless no member clashes there, then the first of 2.5 / 3.5 A at which one does (reported).  The
card's name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.bench_inpaint import gpu_info  # noqa: E402

SAMPLERS = [("ddpm100", "ddpm", 100), ("ddim25", "ddim", 25)]


def timed(fn, n, flush):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        flush.fill_(1)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def summary(t):
    return {"ms_median": statistics.median(t), "ms_min": min(t), "ms_max": max(t), "n": len(t)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5, help="rounds; every round times every pass variant (at least 3)")
    ap.add_argument("--passes", type=int, default=10, help="timed passes of one variant per round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=50, help="timed clash calls per geometry and grow")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_repair.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from codlad_b200 import sampler, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    dsd = weights.init_denoiser_state(0)

    # (1) the clash launches on decoded samples (10 DDPM steps: the launches see only the geometry)
    launches = {}
    for cfg in ("c2", "c4"):
        wl = bench.WORKLOADS[cfg]
        _, _, fs = bench._workload(0, cfg)
        vsd = weights.init_vae_decode_state(0, angle_variant=wl["vae"] in ("K3", "K4"))
        bm = sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=10, precision="f16")
        plan = bm.upload(fs)
        xyz = bm.sample(plan, fs, generator=gen)["xyz"]
        rec = {"residues": fs.NB * fs.L, "atoms": fs.total_atoms, "K": plan.K}
        for thr in (1.2, 2.5):
            for grow in (0, 8):
                for _ in range(args.warmup):
                    bm.residue_clashes(plan, fs, xyz, thr, grow)
                l0 = plan.launches
                t = timed(lambda: bm.residue_clashes(plan, fs, xyz, thr, grow), args.calls, flush)
                counts, keep = bm.residue_clashes(plan, fs, xyz, thr, grow)
                rec[f"thr{thr}_grow{grow}"] = dict(summary(t), launches_per_call=(plan.launches - l0) / args.calls,
                                                   clashing_residues=int((counts > 0).sum()), resampled_residues=int((~keep).sum()))
        launches[cfg] = rec
        del bm, plan, xyz
        torch.cuda.empty_cache()

    # (2) one repair round against a plain pass at configs[1]
    wl = bench.WORKLOADS["c2"]
    _, _, fs = bench._workload(0, "c2")
    vsd = weights.init_vae_decode_state(0)
    bms, plans, inputs, thresholds = {}, {}, {}, {}
    for name, kind, steps in SAMPLERS:
        for mode in ("plain", "repair"):
            bm = sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=steps, precision="f16", sampler=kind)
            bms[(name, mode)], plans[(name, mode)] = bm, bm.upload(fs)
        bm, plan = bms[(name, "repair")], plans[(name, "repair")]
        out = {k: v.clone() for k, v in bm.sample(plan, fs, generator=gen).items()}
        for thr in (1.2, 2.5, 3.5):
            if int(bm.residue_clashes(plan, fs, out["xyz"], thr)[0].sum()) > 0:
                break
        inputs[name], thresholds[name] = out, thr

    def run(name, mode):
        bm, plan = bms[(name, mode)], plans[(name, mode)]
        if mode == "plain":
            return bm.sample(plan, fs, generator=gen)
        return bm.repair(plan, fs, inputs[name], max_rounds=1, threshold=thresholds[name], generator=gen)

    variants = [(name, mode) for name, _, _ in SAMPLERS for mode in ("plain", "repair")]
    for v in variants:
        for _ in range(args.warmup):
            run(*v)
    torch.cuda.synchronize()
    times = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:                               # variants alternate inside every round
            times[v] += timed(lambda: run(*v), args.passes, flush)

    rounds = {}
    for name, kind, steps in SAMPLERS:
        res = run(name, "repair")
        rounds[name] = {"sampler": kind, "steps": steps, "threshold": thresholds[name],
                        "clash_pairs_before_after": res["clash_pairs"].tolist(),
                        "plain_pass": summary(times[(name, "plain")]), "repair_round": summary(times[(name, "repair")]),
                        "round_over_pass": statistics.median(times[(name, "repair")]) / statistics.median(times[(name, "plain")])}
    c2_call = launches["c2"]["thr1.2_grow0"]["ms_median"]
    print(json.dumps({
        "metric": "clash launches of cb2_plan_residue_clashes; one Backmapper.repair round vs Backmapper.sample", "unit": "ms",
        "gpu": gpu_info(), "precision": "f16 (tcgen05, fp32 accumulate)", "weights": "random init (seed 0)",
        "l2": "flushed before every timed call or pass (512 MiB fill)",
        "clash_launches": {"configs[1] (c2: 300 x 10, N6)": launches["c2"], "configs[3] (c4: 2000 x 32, K4, K 48)": launches["c4"]},
        "clash_call_over_ddpm100_pass_c2": c2_call / statistics.median(times[("ddpm100", "plain")]),
        "repair_round_c2": rounds, "rounds": args.rounds, "passes_per_round": args.passes,
    }))


if __name__ == "__main__":
    main()
