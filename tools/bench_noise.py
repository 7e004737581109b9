"""Keyed sampling noise (engine.keyed_normal, Backmapper.sample(seed=...)).  Prints one JSON line with:

  * device time of one keyed fill of 101 slices (the start draw and 100 steps of noise) at configs[1] (10 members x 300 residues)
    and configs[3] (32 members x 2000 residues), CUDA events, L2 overwritten before every fill;
  * device time of one backmapping pass (sampling loop + decode) at configs[1], f16 tier, seeded against generator-drawn noise, for
    DDPM-100 and DDIM-25 (eta = 0), variants alternating in every round, one plan per variant so that no timed pass re-captures;
  * the largest latent difference between a member sampled alone and the same member in the configs[1] batch (same seed and key),
    for both tiers, with the VQ indices that differ and whether the latents came out bit-identical.

    python tools/bench_noise.py [--rounds 3] [--passes 10] [--fills 50] [--warmup 3]

The card's name and power limit are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEED = 0x5EED
SAMPLERS = [("ddpm100", "ddpm", 100), ("ddim25", "ddim", 25)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="rounds; every round times every variant (at least 3)")
    ap.add_argument("--passes", type=int, default=10, help="timed passes of one variant per round")
    ap.add_argument("--fills", type=int, default=50, help="timed fills per configuration")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if not torch.cuda.is_available():
        raise SystemExit("bench_noise.py needs a CUDA device: codlad_b200 has no CPU fallback")
    import bench
    from bench_inpaint import gpu_info
    from codlad_b200 import engine, sampler, synthetic, weights

    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    # ---- the fill alone ----------------------------------------------------------------------------------------------------------
    fills = {}
    for label, name in (("configs[1]", "c2"), ("configs[3]", "c4")):
        w = bench.WORKLOADS[name]
        NB, L = w["ensemble"], w["L"]
        keys = torch.arange(NB, dtype=torch.int64, device=dev)
        out = torch.empty(101, NB, L, 3, device=dev)
        for _ in range(args.warmup):
            engine.keyed_normal(SEED, keys, L, 0, 0, 101, out=out)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.fills)]
        for a, b in ev:
            flush.fill_(1)
            a.record()
            engine.keyed_normal(SEED, keys, L, 0, 0, 101, out=out)
            b.record()
        torch.cuda.synchronize()
        t = [a.elapsed_time(b) * 1e3 for a, b in ev]
        nbytes = out.numel() * 4
        med = statistics.median(t)
        fills[label] = {"members": NB, "residues": L, "slices": 101, "values": out.numel(), "us_median": med, "us_min": min(t),
                        "us_max": max(t), "write_GB_per_s": nbytes / (med * 1e-6) / 1e9}
        del out

    # ---- seeded against generator passes ------------------------------------------------------------------------------------------
    wl = bench.WORKLOADS["c2"]
    prot, batch, fs = bench._workload(0, "c2")
    dsd, vsd = weights.init_denoiser_state(0), weights.init_vae_decode_state(0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    make = lambda kind, T, precision="f16": sampler.Backmapper(dsd, vsd, wl["vae"], k_neighbors=wl["k"], num_sampling_steps=T,
                                                               precision=precision, sampler=kind)
    bms, plans = {}, {}
    for name, kind, T in SAMPLERS:
        for noise in ("generator", "seed"):
            bm = make(kind, T)
            bms[(name, noise)], plans[(name, noise)] = bm, bm.upload(fs)

    def run(name, noise):
        bm, plan = bms[(name, noise)], plans[(name, noise)]
        return bm.sample(plan, fs, generator=gen) if noise == "generator" else bm.sample(plan, fs, seed=SEED)

    variants = list(bms)
    for v in variants:
        for _ in range(args.warmup):
            run(*v)
    torch.cuda.synchronize()
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
    passes = {}
    for name, kind, T in SAMPLERS:
        gen_med = statistics.median(times[(name, "generator")])
        for noise in ("generator", "seed"):
            t = times[(name, noise)]
            med = statistics.median(t)
            passes[f"{name}_{noise}"] = {"sampler": kind, "T": T, "ms_per_pass_median": med, "ms_per_pass_min": min(t),
                                         "ms_per_pass_max": max(t), "residues_per_s": fs.NB * fs.L / (med * 1e-3),
                                         "over_generator_time": med / gen_med,
                                         "plan_launches_per_pass": statistics.median(launches[(name, noise)])}
    del bms, plans
    torch.cuda.empty_cache()

    # ---- a member alone against the batch ----------------------------------------------------------------------------------------
    batching = {}
    for precision in ("fp32", "f16"):
        bm = make("ddpm", 100, precision)
        keys = sampler.member_keys(fs)
        res = bm.sample(bm.upload(fs), fs, seed=SEED)
        lat, idx = res["latent"].clone(), res["idx"].clone()
        one = sampler.frames_from_batch(batch, prot.info, 1)
        worst, flips, identical = 0.0, 0, 0
        for b in range(fs.NB):
            alone = bm.sample(bm.upload(one), one, seed=SEED, keys=keys[b:b + 1])
            worst = max(worst, float((alone["latent"][0] - lat[b]).abs().max()))
            flips += int((alone["idx"][0] != idx[b]).sum())
            identical += int(torch.equal(alone["latent"][0], lat[b]))
        batching[precision] = {"configs[1]": {"members": fs.NB, "residues": fs.L, "sampler": "ddpm100",
                                              "max_abs_latent_difference": worst, "latent_abs_max": float(lat.abs().max()),
                                              "vq_flips": flips, "vq_rows": fs.NB * fs.L, "bit_identical_members": identical}}
        # ragged: frames of 80 / 70 / 40 residues, 4 members, each member alone on its own frame at its own length (unpadded)
        prots = [synthetic.make_protein(n, 1, seed=500 + 7 * i + n) for i, n in enumerate((80, 70, 40))]
        frame_of = [0, 1, 2, 1]
        rfs = sampler.frames_from_batch(synthetic.collate_many(prots), [p.info for p in prots], frame_of=frame_of)
        rkeys = sampler.member_keys(rfs)
        res = bm.sample(bm.upload(rfs), rfs, seed=SEED)
        lat, idx = res["latent"].clone(), res["idx"].clone()
        rows = []
        for b, f in enumerate(frame_of):
            n = prots[f].L
            one = sampler.frames_from_batch(synthetic.collate(prots[f]), prots[f].info, 1)
            alone = bm.sample(bm.upload(one), one, seed=SEED, keys=rkeys[b:b + 1])
            d = (alone["latent"][0] - lat[b, :n]).abs()
            rows.append({"member": b, "residues": n, "padded_in_batch_to": rfs.L, "max_abs_latent_difference": float(d.max()),
                         "rel_err": float((alone["latent"][0] - lat[b, :n]).norm() / lat[b, :n].norm()),
                         "rows_differing": int((d.amax(-1) > 0).sum()),
                         "vq_flips": int((alone["idx"][0] != idx[b, :n]).sum()),
                         "bit_identical": bool(torch.equal(alone["latent"][0], lat[b, :n]))})
        batching[precision]["ragged_unpadded_alone"] = rows
        del bm
        torch.cuda.empty_cache()

    print(json.dumps({
        "metric": "keyed sampling noise: engine.keyed_normal fill time, seeded against generator passes, batch invariance",
        "gpu": gpu_info(), "weights": "random init (seed 0)",
        "fill": {"unit": "us per fill of 101 slices [101, NB, L, 3] float32, CUDA events",
                 "l2": "flushed before every fill (512 MiB fill)", "fills": args.fills, "configs": fills},
        "passes": {"workload": "configs[1]: PED-like 300-residue IDP, N6, num_ensemble=10", "precision": "f16 (tcgen05, fp32 accumulate)",
                   "unit": "ms per pass (sampling loop + decode), CUDA events", "l2": "flushed before every timed pass (512 MiB fill)",
                   "rounds": args.rounds, "passes_per_round": args.passes, "variants": passes},
        "member_alone_vs_batch": {"note": "each member sampled alone on its frame with its own key against the batch, DDPM-100: "
                                          "configs[1] (one 300-residue frame, same L alone), and a ragged 80/70/40 batch whose "
                                          "members are sampled alone at their own, unpadded length",
                                  "tiers": batching},
    }))


if __name__ == "__main__":
    main()
