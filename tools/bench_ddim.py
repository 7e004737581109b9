"""DDIM vs DDPM at configs[1] (one 300-residue frame x 10 members, N6 decoder, f16 tier): device time per backmapping pass
(sampling loop + decode) of DDPM-100 and of DDIM eta = 0 at 100, 50 and 25 steps, run alternately in one process, plus the
DDIM-25 latent of the f16 tier against the fp32 tier.  Prints one JSON line.

    python tools/bench_ddim.py [--rounds 5] [--passes 10] [--warmup 3]

Each timed pass is bracketed by CUDA events with the L2 overwritten (512 MiB fill) before it, as bench.py does.  The card's
name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

VARIANTS = [("ddpm100", "ddpm", 100), ("ddim100", "ddim", 100), ("ddim50", "ddim", 50), ("ddim25", "ddim", 25)]


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
        raise SystemExit("bench_ddim.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from codlad_b200 import sampler, synthetic, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    wl = bench.WORKLOADS["c2"]
    _, _, fs = bench._workload(0, "c2")
    fs.pin()
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)

    def backmapper(kind, steps, precision="f16"):
        return sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=steps, precision=precision, sampler=kind)

    bms = {name: backmapper(kind, steps) for name, kind, steps in VARIANTS}
    plans = {name: bm.upload(fs) for name, bm in bms.items()}
    gen = torch.Generator(device=dev).manual_seed(1234)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    for name, bm in bms.items():
        for _ in range(args.warmup):
            bm.sample(plans[name], fs, generator=gen)
    torch.cuda.synchronize()

    times = {name: [] for name in bms}
    launches = {name: [] for name in bms}
    for _ in range(args.rounds):
        for name, bm in bms.items():                     # variants alternate inside every round
            plan = plans[name]
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.passes)]
            l0 = plan.launches
            for a, b in ev:
                flush.fill_(1)
                a.record()
                bm.sample(plan, fs, generator=gen)
                b.record()
            torch.cuda.synchronize()
            times[name] += [a.elapsed_time(b) for a, b in ev]
            launches[name].append((plan.launches - l0) / args.passes)

    residues = fs.NB * fs.L
    out = {}
    for name, kind, steps in VARIANTS:
        med = statistics.median(times[name])
        out[name] = {"sampler": kind, "eta": 0.0 if kind == "ddim" else None, "steps": steps, "ms_per_pass_median": med,
                     "ms_per_pass_min": min(times[name]), "ms_per_pass_max": max(times[name]), "residues_per_s": residues / (med * 1e-3),
                     "launches_per_pass": statistics.median(launches[name])}

    # the DDIM-25 latent of the f16 tier against the fp32 tier, same initial noise
    z = synthetic.latent_noise((fs.NB, fs.L, 3), 7)
    bm32 = backmapper("ddim", 25, "fp32")
    o16 = bms["ddim25"].sample(plans["ddim25"], fs, z)
    lat16, idx16 = o16["latent"].clone(), o16["idx"].clone()
    o32 = bm32.sample(bm32.upload(fs), fs, z)
    lat32 = o32["latent"].double()
    tiers = {"latent_rel_err": float((lat16.double() - lat32).norm() / lat32.norm()),
             "vq_flip_rate": float((idx16 != o32["idx"]).float().mean())}

    print(json.dumps({
        "metric": "backmapping pass, DDIM (eta = 0) vs DDPM", "unit": "ms per pass / residues/s", "gpu": gpu_info(),
        "workload": "configs[1]: PED-like 300-residue IDP, N6, num_ensemble=10", "precision": "f16 (tcgen05, fp32 accumulate)", "residues_per_pass": residues,
        "weights": "random init (seed 0)", "l2": "flushed before every timed pass (512 MiB fill)",
        "rounds": args.rounds, "passes_per_round": args.passes, "variants": out,
        "ddim25_over_ddpm100_residues_per_s": out["ddim25"]["residues_per_s"] / out["ddpm100"]["residues_per_s"],
        "ddim25_f16_vs_fp32": tiers,
    }))


if __name__ == "__main__":
    main()
