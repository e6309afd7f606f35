"""Cost of the posterior draws (lapf_sampler_draws_enable): device time per step with them off and on.

    python tools/draws_probe.py [--steps N] [--rounds R] [--out FILE]

Two shapes, as in tools/batch_means_probe.py: the benchmark's (65,536 walkers over 100 epochs, 64x64
stamps, 2-body, 128 updates per step) and the reference's (24 walkers, 16 warps per walker, 128-pixel
stamp, whole-frame domain), each at thin 16 and thin 1, draws off and on (64 per walker), sketches on
as on the command line.  No chain is recorded: this is what a --no-chains --draws run pays for.
Device times are CUDA events around the sampler's launches, the configurations alternated over
--rounds rounds (medians reported).  Card name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from batch_means_probe import time_steps  # noqa: E402
from chain_events_probe import benchmark_shape, card, reference_shape  # noqa: E402
from olpefit_b200 import sampler  # noqa: E402

K = 64


def make(shape, thin, draws):
    dom, init, frame_of, team = shape
    s = sampler.GibbsSampler(dom, init, frame_of, seed=11, burn_in=0, thin=thin, team_warps=team)
    s.enable_sketch()
    if draws:
        s.enable_draws(K)
    return s


def measure(shape_fn, U, steps, rounds):
    shape = shape_fn()
    samplers = {(thin, dr): make(shape, thin, dr) for thin in (16, 1) for dr in (False, True)}
    times = {k: [] for k in samplers}
    for _ in range(rounds):
        for k, s in samplers.items():
            times[k].append(time_steps(s, U, steps))
    out = []
    for (thin, dr), t in times.items():
        res = {"thin": thin, "draws": K if dr else "off", "device_ms_per_step": float(np.median(t)),
               "rounds_ms": [round(v, 4) for v in t]}
        print(json.dumps(res), flush=True)
        out.append(res)
    for thin in (16, 1):
        off = float(np.median(times[thin, False]))
        print("thin %d: draws cost %+.2f %%" % (thin, 100.0 * (float(np.median(times[thin, True])) / off - 1.0)), flush=True)
    for s in samplers.values():
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU")
    torch.cuda.set_device(0)
    result = {"card_before": card(), "updates_per_step": 128, "per_walker": K}
    print(result["card_before"], flush=True)
    print("benchmark shape: 65536 walkers x 100 epochs, 64x64, 2-body", flush=True)
    result["benchmark"] = measure(benchmark_shape, 128, args.steps, args.rounds)
    print("reference shape: 24 walkers, team 16, 128-pixel stamp, whole-frame domain", flush=True)
    result["reference"] = measure(reference_shape, 128, args.steps, args.rounds)
    result["card_after"] = card()
    print(result["card_after"], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
