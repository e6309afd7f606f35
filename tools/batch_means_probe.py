"""Cost of the batch means (lapf_sampler_batchmeans_enable): device time per step with them off and on.

    python tools/batch_means_probe.py [--steps N] [--out FILE]

Two shapes, as in tools/chain_events_probe.py: the benchmark's (65,536 walkers over 100 epochs, 64x64
stamps, 2-body, 128 updates per step) at thin 16 and thin 1, each with batch_rows 1 (every recorded row
closes a batch: the worst case), 64 (the command line's setting) and 2^20 (no row of the run closes a
batch: what the per-row test alone costs), sketches on as on the command line;
and the reference's (24 walkers, 16 warps per walker, 128-pixel stamp, whole-frame domain) at thin 1.
No chain is recorded: the moments, sketches and batch means are what a --no-chains run pays for.
Device times are CUDA events around the sampler's launches, the configurations alternated over
--rounds rounds.  Card name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from chain_events_probe import benchmark_shape, card, reference_shape  # noqa: E402
from olpefit_b200 import sampler  # noqa: E402

LEVELS = 16


def make(shape, thin, batch_rows):
    dom, init, frame_of, team = shape
    s = sampler.GibbsSampler(dom, init, frame_of, seed=11, burn_in=0, thin=thin, team_warps=team)
    s.enable_sketch()
    if batch_rows:
        s.enable_batch_means(batch_rows, LEVELS)
    return s


def time_steps(s, U, steps):
    s.run(U, record=False)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        s.run(U, record=False)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def measure(shape_fn, configs, U, steps, rounds):
    shape = shape_fn()
    samplers = {(thin, br): make(shape, thin, br) for thin, br in configs}
    times = {k: [] for k in samplers}
    for _ in range(rounds):
        for k, s in samplers.items():
            times[k].append(time_steps(s, U, steps))
    out = []
    for (thin, br), t in times.items():
        res = {"thin": thin, "batch_rows": br or "off", "device_ms_per_step": float(np.median(t)),
               "rounds_ms": [round(v, 4) for v in t]}
        print(json.dumps(res), flush=True)
        out.append(res)
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
    result = {"card_before": card(), "updates_per_step": 128, "levels": LEVELS}
    print(result["card_before"], flush=True)
    print("benchmark shape: 65536 walkers x 100 epochs, 64x64, 2-body", flush=True)
    result["benchmark"] = measure(benchmark_shape, [(t, b) for t in (16, 1) for b in (0, 1, 64, 1 << 20)], 128, args.steps,
                                  args.rounds)
    print("reference shape: 24 walkers, team 16, 128-pixel stamp, whole-frame domain", flush=True)
    result["reference"] = measure(reference_shape, [(1, 0), (1, 1), (1, 64)], 128, args.steps, args.rounds)
    result["card_after"] = card()
    print(result["card_after"], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
