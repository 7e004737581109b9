"""Latent inpainting vs a plain pass at configs[1] (one 300-residue frame x 10 members, N6 decoder, f16 tier): device time per
backmapping pass (sampling loop + decode) of Backmapper.sample against Backmapper.resample with half the residues of every
member kept, for DDPM-100 and DDIM-25 (eta = 0), run alternately in one process; plus the cost of switching one plan
between plain and inpainting passes, each switch re-capturing the step-loop graph.  Prints one JSON line.

    python tools/bench_inpaint.py [--rounds 5] [--passes 10] [--warmup 3]

Each timed pass is bracketed by CUDA events with the L2 overwritten (512 MiB fill) before it, as bench.py does.  The card's
name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SAMPLERS = [("ddpm100", "ddpm", 100), ("ddim25", "ddim", 25)]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        return {"name": torch.cuda.get_device_name(0), "power_limit": None}
    name, power = (v.strip() for v in r.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5, help="rounds; every round times every variant (at least 3)")
    ap.add_argument("--passes", type=int, default=10, help="timed passes of one variant per round")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_inpaint.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from codlad_b200 import sampler, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    wl = bench.WORKLOADS["c2"]
    _, _, fs = bench._workload(0, "c2")
    fs.pin()
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    keep = torch.rand(fs.NB, fs.L, device=dev, generator=gen) < 0.5            # half the residues of every member, scattered

    # per sampler: one Backmapper and one plan for plain passes, one of each for inpainting passes (no re-capture inside a
    # timed variant), and a third plan that switches between the two kinds of pass
    bms, plans, latents = {}, {}, {}
    for name, kind, steps in SAMPLERS:
        for mode in ("plain", "inpaint", "switch"):
            bm = sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=steps, precision="f16", sampler=kind)
            bms[(name, mode)], plans[(name, mode)] = bm, bm.upload(fs)
        bm, plan = bms[(name, "inpaint")], plans[(name, "inpaint")]
        latents[name] = bm.sample(plan, fs, generator=gen)["latent"].clone()

    def run(name, mode):
        bm, plan = bms[(name, mode)], plans[(name, mode)]
        if mode == "plain":
            return bm.sample(plan, fs, generator=gen)
        return bm.resample(plan, fs, latents[name], keep, generator=gen)

    variants = [(name, mode) for name, _, _ in SAMPLERS for mode in ("plain", "inpaint")]
    for v in variants:
        for _ in range(args.warmup):
            run(*v)
    torch.cuda.synchronize()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    times = {v: [] for v in variants}
    launches = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:                               # variants alternate inside every round
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

    # one plan alternating plain and inpainting passes: every switch re-captures the step-loop graph.  Host wall time of a
    # synchronised pass, against the same on the plans that never switch.
    def wall(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    def switch_pass(name, i):
        bm, plan = bms[(name, "switch")], plans[(name, "switch")]
        if i % 2 == 0:
            bm.sample(plan, fs, generator=gen)
        else:
            bm.resample(plan, fs, latents[name], keep, generator=gen)

    switching = {}
    n_switch = max(2 * args.rounds, 6)
    for name, _, _ in SAMPLERS:
        alt = [wall(lambda: switch_pass(name, i)) for i in range(n_switch)]
        fixed = [wall(lambda: run(name, mode)) for mode in ("plain", "inpaint") for _ in range(n_switch // 2)]
        switching[name] = {"alternating_ms_per_pass_median": statistics.median(alt),
                           "non_switching_ms_per_pass_median": statistics.median(fixed),
                           "recapture_ms_per_switch": statistics.median(alt) - statistics.median(fixed), "passes": n_switch}

    residues = fs.NB * fs.L
    out = {}
    for name, kind, steps in SAMPLERS:
        for mode in ("plain", "inpaint"):
            t = times[(name, mode)]
            med = statistics.median(t)
            out[f"{name}_{mode}"] = {"sampler": kind, "steps": steps, "call": "sample" if mode == "plain" else "resample",
                                     "ms_per_pass_median": med, "ms_per_pass_min": min(t), "ms_per_pass_max": max(t),
                                     "residues_per_s": residues / (med * 1e-3),
                                     "launches_per_pass": statistics.median(launches[(name, mode)])}
        out[f"{name}_inpaint_over_plain_time"] = out[f"{name}_inpaint"]["ms_per_pass_median"] / out[f"{name}_plain"]["ms_per_pass_median"]

    print(json.dumps({
        "metric": "backmapping pass, Backmapper.resample (half the residues kept) vs Backmapper.sample", "unit": "ms per pass",
        "gpu": gpu_info(), "workload": "configs[1]: PED-like 300-residue IDP, N6, num_ensemble=10",
        "precision": "f16 (tcgen05, fp32 accumulate)", "residues_per_pass": residues, "kept_fraction": float(keep.float().mean()),
        "weights": "random init (seed 0)", "l2": "flushed before every timed pass (512 MiB fill)",
        "rounds": args.rounds, "passes_per_round": args.passes, "variants": out,
        "plain_inpaint_switching_host_wall_clock": switching,
    }))


if __name__ == "__main__":
    main()
