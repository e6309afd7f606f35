"""Cost and benefit of per-epoch jump widths (lapf_sampler_set_frame_widths / adapt_widths).

    python tools/frame_widths_probe.py [--steps N] [--rounds R] [--out FILE]

Cost: device time per step with the table off and on (every row the batch widths, so the chains are the
same), at the benchmark's shape (65,536 walkers over 100 epochs, 64x64 stamps, 2-body, 128 updates per
step) and the reference's (24 walkers, 16 warps per walker, 128-pixel stamp, whole-frame domain), each at
thin 16 and thin 1, sketches on as on the command line, no chain recorded.  Then the adaptation step per
window at both shapes: frame_counts, the all-reduce (one rank: nothing to add) and adapt_widths.  Device
times are CUDA events, the configurations alternated over --rounds rounds (medians reported).

Benefit: three epochs whose objects are 0.25x, 1x and 4x as bright (at 1x a 4000-count star and a 1000-count
companion), 64 walkers
each, run through the command line with --mcse --no-chains and the same burn-in and stop rule three times:
fixed widths, --adapt and --adapt-per-epoch.  Reported per epoch: the separation and position-angle ESS
per recorded row, and the post-burn-in acceptance of the positions.  Card name, power limit and SM clock
are read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from batch_means_probe import time_steps  # noqa: E402
from chain_events_probe import benchmark_shape, card, reference_shape  # noqa: E402
from olpefit_b200 import chains, cli, dist, frame, sampler, synth  # noqa: E402

SCALES = (0.25, 1.0, 4.0)


def make(shape, thin, table):
    dom, init, frame_of, team = shape
    s = sampler.GibbsSampler(dom, init, frame_of, seed=11, burn_in=0, thin=thin, team_warps=team)
    s.enable_sketch()
    if table:
        s.set_frame_widths()
    return s


def time_adapt(s, reps):
    """Device ms of one adaptation step (frame_counts, all-reduce, adapt_widths)."""
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        s.adapt_widths(dist.allreduce_sum(s.frame_counts()), 0.35)
    t0.record()
    for _ in range(reps):
        s.adapt_widths(dist.allreduce_sum(s.frame_counts()), 0.35)
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / reps


def measure(shape_fn, U, steps, rounds):
    shape = shape_fn()
    samplers = {(thin, tb): make(shape, thin, tb) for thin in (16, 1) for tb in (False, True)}
    times = {k: [] for k in samplers}
    for _ in range(rounds):
        for k, s in samplers.items():
            times[k].append(time_steps(s, U, steps))
    out = {"steps": []}
    for (thin, tb), t in times.items():
        res = {"thin": thin, "table": "on" if tb else "off", "device_ms_per_step": float(np.median(t)),
               "rounds_ms": [round(v, 4) for v in t]}
        print(json.dumps(res), flush=True)
        out["steps"].append(res)
    for thin in (16, 1):
        off = float(np.median(times[thin, False]))
        print("thin %d: table on %+.2f %%" % (thin, 100.0 * (float(np.median(times[thin, True])) / off - 1.0)), flush=True)
    out["adapt_ms_per_window"] = time_adapt(samplers[16, True], 200)
    print("adaptation step: %.4f ms" % out["adapt_ms_per_window"], flush=True)
    for s in samplers.values():
        s.close()
    return out


def write_epochs(tmp):
    paths = []
    for f, a in enumerate(SCALES):
        d = os.path.join(tmp, "epoch%d" % f)
        os.makedirs(d)
        p = synth.truth_parameters(2, f)
        p[6:8] = a * np.array([4000.0, 1000.0])
        rng = np.random.default_rng(300 + f)
        t = synth.truth_image(p, 2, (0, 1024, 0, 1024))
        img = rng.poisson(t + synth.SKY_LEVEL).astype(np.float64) - synth.SKY_LEVEL + rng.normal(0, synth.READ_NOISE, t.shape)
        path = os.path.join(d, "N2.2009053%d.2996%d.LDIF.fits" % (f, f))
        frame.write_fits(path, img.astype(np.float32), synth.HEADER)
        os.makedirs(chains.results_dir(path))
        chains.write_walker_csv(chains.results_dir(path) + "step2a.csv", np.concatenate([p, [0.0]])[None])
        paths.append(path)
    lst = os.path.join(tmp, "frames.txt")
    with open(lst, "w") as fh:
        fh.write("\n".join(paths[1:]) + "\n")
    return paths, lst


def benefit(walkers, burn_in, accept_min):
    out = {}
    for mode, flags in (("fixed", []), ("adapt", ["--adapt"]), ("adapt_per_epoch", ["--adapt-per-epoch"])):
        with tempfile.TemporaryDirectory() as tmp:
            paths, lst = write_epochs(tmp)
            argv = [paths[0], "-i", "2a", "--frames", lst, "--walkers", str(walkers), "--burn-in", str(burn_in),
                    "--accept-min", str(accept_min), "--seed", "41", "--stamp", "64", "--mcse", "--no-chains",
                    "--quiet"] + flags
            cli.main_step2(argv)
            rows = []
            for f, path in enumerate(paths):
                s = json.load(open(chains.results_dir(path) + "step2_summary.json"))
                c = s["sep_pa_companion"]
                n = c["rows"]
                rows.append({"scale": SCALES[f], "updates": s["updates"], "rows": n,
                             "sep_ess": c["sep_mas"]["ess"], "pa_ess": c["pa_deg"]["ess"],
                             "sep_ess_per_row": c["sep_mas"]["ess"] / n, "pa_ess_per_row": c["pa_deg"]["ess"] / n,
                             "acceptance": s.get("acceptance"),
                             "widths": s.get("widths")})
                print(mode, json.dumps({k: v for k, v in rows[-1].items() if k not in ("acceptance", "widths")}),
                      flush=True)
            out[mode] = rows
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--walkers", type=int, default=64, help="walkers per epoch in the benefit run")
    ap.add_argument("--burn-in", type=int, default=6144)
    ap.add_argument("--accept-min", type=int, default=1500)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU")
    torch.cuda.set_device(0)
    result = {"card_before": card(), "updates_per_step": 128}
    print(result["card_before"], flush=True)
    print("benchmark shape: 65536 walkers x 100 epochs, 64x64, 2-body", flush=True)
    result["benchmark"] = measure(benchmark_shape, 128, args.steps, args.rounds)
    print("reference shape: 24 walkers, team 16, 128-pixel stamp, whole-frame domain", flush=True)
    result["reference"] = measure(reference_shape, 128, args.steps, args.rounds)
    print("benefit: epochs at %s x brightness, %d walkers each" % (SCALES, args.walkers), flush=True)
    result["benefit"] = {"walkers_per_epoch": args.walkers, "burn_in": args.burn_in, "accept_min": args.accept_min,
                         "modes": benefit(args.walkers, args.burn_in, args.accept_min)}
    result["card_after"] = card()
    print(result["card_after"], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
