"""Cost of recording every update (thin = 1): device time and bytes per step of the dense chain formats
and the chain events (LAPF_CHAIN_EVENTS_*), the ChainStreamer's end-to-end time per step into pinned
memory, and the host decode time per step.

    python tools/chain_events_probe.py [--steps N] [--out FILE]

Two shapes: the benchmark's (65,536 walkers over 100 epochs, 64x64 stamps, 2-body, 128 updates per
step) and the reference's (24 walkers, 16 warps per walker, 128-pixel stamp with the whole-frame
domain of a 1024x1024 frame).  'none' runs record no chain, but still accumulate the moments (and at
thin = 1 that is 2(P+1) FP64 reductions per update); 'none thin 16' is the benchmark's setting.
Device times are CUDA events around the sampler's launches; the streamer's time is a host clock over
N segments that ends in a synchronise.  Card name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from olpefit_b200 import chains, frame, sampler, synth  # noqa: E402

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}
FORMATS = [("none thin 16", None, 16), ("none", None, 1), ("dense f32", "f32delta", 1), ("events f32", "events_f32delta", 1),
           ("dense f64", "f64", 1), ("events f64", "events_f64", 1)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def benchmark_shape():
    W, F, S = 65536, 100, 64
    stamps, origins = synth.make_stamps(F, S, 2)
    dom = frame.prepare_domain(stamps, HEADER, origin=origins, nbody=2)
    frame_of = (np.arange(W) % F).astype(np.int32)
    p0 = frame.initial_parameters(stamps[0], synth.step1_guess(stamps[0], 2, origin=tuple(origins[0])), 2,
                                  origin=tuple(origins[0]))
    return dom, np.tile(p0, (W, 1)), frame_of, 1


def reference_shape():
    img, truth = synth.make_frame(0, 2)
    cut = frame.stamp_cut(truth, 2, 128, img.shape)
    dom = frame.prepare_domain(img, HEADER, size=128, cut=cut, nbody=2, whole_frame=True)
    guess = synth.step1_guess(img, 2, sky_xy=(100, 120))
    p0 = frame.initial_parameters(img, guess, 2)
    return dom, np.tile(p0, (24, 1)), None, 16


def measure(shape_fn, U, steps):
    dom, init, frame_of, team = shape_fn()
    out = []
    for name, fmt, thin in FORMATS:
        s = sampler.GibbsSampler(dom, init, frame_of, seed=11, burn_in=0, thin=thin, team_warps=team)
        if fmt:
            s.set_chain_format(fmt)
        nbytes = s.chain_bytes(U) if fmt else 0
        buf = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=dom.device)

        def step():
            if fmt is None:
                s.run(U, record=False)
            elif s.events:
                s.run(U, out=buf)
            else:
                s.run(U, out=buf.view(s.chain_dtype))
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            step()
        t1.record()
        torch.cuda.synchronize()
        res = {"format": name, "thin": thin, "device_ms_per_step": t0.elapsed_time(t1) / steps, "bytes_per_step": nbytes}
        if fmt:
            st = sampler.ChainStreamer(s, U)
            st.run(U)
            st.run(U)
            torch.cuda.synchronize()
            h0 = time.perf_counter()
            for _ in range(steps):
                seg = st.run(U)
            last = st.finish()
            res["streamer_ms_per_step"] = 1e3 * (time.perf_counter() - h0) / steps
            if s.events:
                raw, rows = last
                h0 = time.perf_counter()
                dec = chains.decode_events(raw, rows, s.n_walkers, s.nparam + 1, np.float32 if "f32" in name else np.float64)
                res["host_decode_ms_per_step"] = 1e3 * (time.perf_counter() - h0)
                res["decoded_bytes"] = int(dec.nbytes)
            del st, seg, last
        s.close()
        out.append(res)
        print(json.dumps(res), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU")
    torch.cuda.set_device(0)
    result = {"card_before": card()}
    print(result["card_before"], flush=True)
    print("benchmark shape: 65536 walkers x 100 epochs, 64x64, 2-body, 128 updates per step", flush=True)
    result["benchmark"] = measure(benchmark_shape, 128, args.steps)
    print("reference shape: 24 walkers, team 16, 128-pixel stamp, whole-frame domain, 128 updates per step", flush=True)
    result["reference"] = measure(reference_shape, 128, args.steps)
    result["card_after"] = card()
    print(result["card_after"], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
