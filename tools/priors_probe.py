"""Cost of parameter priors (lapf_sampler_set_priors).

    python tools/priors_probe.py [--steps N] [--rounds R] [--out FILE]

Device time per step, CUDA events, with the configurations alternated over --rounds rounds (medians
reported), at the benchmark's shape (65,536 walkers over 100 epochs, 64x64 stamps, 2-body, batched kernel)
and the reference's (24 walkers, 16 warps per walker, 128-pixel stamp, whole-frame domain), 128 updates per
step, thin 16, sketches on as on the command line, no chain recorded:
  off      no table
  neutral  every box infinite and every sigma +inf (the chains of `off`, bit for bit)
  gauss    a Gaussian term on every parameter (mu the start, sigma ten jump widths), no box
  box      a box on every parameter around the start, 3 jump widths each way
Each line also gives the acceptance and `skipped`, the share of proposals whose pass the batched kernel
skipped (1 - exponentials evaluated / those of `off`; with the box, the proposals it rejected; the team
kernels evaluate them all).  Card name, power limit and SM clock are read in the same run.
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
from olpefit_b200 import layout, sampler  # noqa: E402

CONFIGS = ("off", "neutral", "gauss", "box")
BOX_WIDTHS = 3.0


def table(kind, dom, init, frame_of):
    F, P = dom.n_frames, init.shape[1]
    t = np.tile([-np.inf, np.inf, 0.0, np.inf], (F, P, 1))
    if kind == "neutral":
        return t
    w, is_log = layout.default_widths(2)
    fo = np.zeros(init.shape[0], dtype=int) if frame_of is None else frame_of
    for f in range(F):
        p = init[np.argmax(fo == f)]
        if kind == "gauss":
            t[f, :, 2] = p
            t[f, :, 3] = 10 * w * np.where(is_log, np.abs(p) * np.log(10.0), 1.0)
        else:
            a = np.where(is_log, p * 10 ** (-BOX_WIDTHS * w), p - BOX_WIDTHS * w)
            b = np.where(is_log, p * 10 ** (BOX_WIDTHS * w), p + BOX_WIDTHS * w)
            t[f, :, 0], t[f, :, 1] = np.minimum(a, b), np.maximum(a, b)
    return t


def make(shape, kind):
    dom, init, frame_of, team = shape
    s = sampler.GibbsSampler(dom, init, frame_of, seed=11, burn_in=0, thin=16, team_warps=team)
    s.enable_sketch()
    if kind != "off":
        t = table(kind, dom, init, frame_of)
        s.set_priors(t[..., 0], t[..., 1], t[..., 2], t[..., 3])
    return s


def measure(shape_fn, U, steps, rounds):
    shape = shape_fn()
    samplers = {k: make(shape, k) for k in CONFIGS}
    times = {k: [] for k in CONFIGS}
    for _ in range(rounds):
        for k, s in samplers.items():
            times[k].append(time_steps(s, U, steps))
    out = {"steps": []}
    off = float(np.median(times["off"]))
    exps_off = None
    for k in CONFIGS:
        st = samplers[k].stats(moments=False)
        exps = float(st["exps"].item()) / float(st["tries"].sum().item())
        exps_off = exps if exps_off is None else exps_off
        res = {"priors": k, "device_ms_per_step": float(np.median(times[k])), "rounds_ms": [round(v, 4) for v in times[k]],
               "vs_off_percent": 100.0 * (float(np.median(times[k])) / off - 1.0),
               "acceptance": float(st["accepts"].sum().item()) / float(st["tries"].sum().item()),
               "exps_per_update": exps, "skipped": 1.0 - exps / exps_off}
        print(json.dumps(res), flush=True)
        out["steps"].append(res)
    for s in samplers.values():
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card_before": card()}
    print(res["card_before"], flush=True)
    res["benchmark_shape"] = measure(benchmark_shape, 128, args.steps, args.rounds)
    res["reference_shape"] = measure(reference_shape, 128, args.steps * 5, args.rounds)
    res["card_after"] = card()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
