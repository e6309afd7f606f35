#!/usr/bin/env python
"""Benchmark of the LAPF step-2 hot path on B200 (see DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] ...               # the reference algorithm on host cores
    python bench.py --dump-outputs DIR ...                        # also write the last timed step's chain rows

Workload (BASELINE.json configs[2], the single-GPU throughput configuration): 65,536 independent
walkers per GPU spread over 100 synthetic NIRC2-like epochs, 64 x 64 stamps, 2-body model.
One "step" = ``--updates-per-step`` Gibbs updates of every walker (default 128 = 8 sweeps of the
16 parameters), recording one chain row per sweep.  Metric: pixel-model evaluations per second
(= Gibbs updates/s x pixels per stamp); Gibbs updates/s is reported next to it.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}
METRIC = "pixel_model_evals_per_sec"
UNIT = "pixel-evals/s"
DUMP_BYTES = 32 << 20           # --dump-outputs: small enough to keep and compare two builds' dumps


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--walkers", type=int, default=65536, help="walkers per GPU")
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--stamp", type=int, default=64, choices=[32, 64, 128])
    ap.add_argument("--nbody", type=int, default=2, choices=[2, 3])
    ap.add_argument("--updates-per-step", type=int, default=128)
    ap.add_argument("--thin", type=int, default=16)
    ap.add_argument("--seed", type=int, default=2019)
    ap.add_argument("--team", type=int, default=1, choices=[1, 4, 16], help="warps per walker (16 for few walkers)")
    ap.add_argument("--cpu-updates", type=int, default=80000, help="updates per CPU walker in the baseline sample")
    ap.add_argument("--ref-updates-per-step", type=int, default=4000, help="updates per CPU walker and step, --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the 1-walker / 64-walker block (BASELINE configs 1-2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the chain rows the last timed step returned (rank 0's walkers, "
                         "float64) to DIR/chain.npy; above %d MiB a sample of walkers drawn with --seed stands for them"
                         % (DUMP_BYTES >> 20))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's chain; --impl reference keeps none")
    return a


def workload_name(a):
    return ("config3: %d walkers/GPU x %d epochs, %dx%d stamps, %d-body, %d updates/step"
            % (a.walkers, a.frames, a.stamp, a.stamp, a.nbody, a.updates_per_step))


def workload_config(a):
    """The keys both arms print, so the two lines describe the same workload."""
    return {"workload": workload_name(a), "walkers_per_gpu": a.walkers, "frames": a.frames, "stamp": a.stamp,
            "nbody": a.nbody, "updates_per_step": a.updates_per_step, "thin": a.thin, "team_warps": a.team,
            "l2": "GPU arm: L2 flushed between timed steps (256 MiB memset outside the event pairs), stamps re-staged "
                  "from HBM into shared memory by TMA in every launch; CPU arm (--impl reference): a bounded sample of "
                  "the same workload on the host cores, no device involved"}


# ----------------------------------------------------------------------------------------------
# CPU side (the reference algorithm through the oracle port; the only place bench.py runs oracle/)
# ----------------------------------------------------------------------------------------------
def _cpu_walker(job):
    """One host walker: the float64 numpy restatement of the reference loop on one stamp."""
    nbody, size, n_updates, seed = job
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    from olpefit_b200 import synth
    from oracle import lapf_oracle as orc
    lay = orc.layout_for(nbody)
    ox, oy = synth.stamp_origin(size, nbody)
    img32, _ = synth.make_frame(0, nbody, region=(oy, oy + size, ox, ox + size))
    img = img32.astype(np.float64)
    w = orc.weight_map(img, HEADER)
    guess = synth.step1_guess(img32, nbody, origin=(ox, oy))
    g_local = guess - np.array([ox, oy] * nbody + [ox, oy], dtype=np.float64)
    p0 = orc.initial_parameters(img, g_local, lay)
    p0[0:2 * nbody:2] += ox
    p0[1:2 * nbody:2] += oy
    t0 = time.perf_counter()
    res = orc.run_chain(img, w, lay, p0, orc.NumpyStream(seed), origin=(ox, oy), n_updates=n_updates, burn_in=0)
    return time.perf_counter() - t0, res.n_updates


def cpu_full_frame(nbody, n_updates):
    """One host walker on the reference's own pixel domain, the whole 1024 x 1024 frame
    (apf_step2.py:94,237): seconds per update on one core."""
    from olpefit_b200 import synth
    from oracle import lapf_oracle as orc
    lay = orc.layout_for(nbody)
    img32, truth = synth.make_frame(0, nbody)
    img = img32.astype(np.float64)
    w = orc.weight_map(img, HEADER)
    t0 = time.perf_counter()
    orc.run_chain(img, w, lay, truth, orc.NumpyStream(1), n_updates=n_updates, burn_in=0)
    return (time.perf_counter() - t0) / (n_updates + 1)      # + the initial evaluation


def cpu_walkers(nbody, size, n_updates, cores):
    """``cores`` walkers in ``cores`` processes (one process per walker, like one MPI rank per
    walker, apf_step2.py:54-57).  Returns (seconds of the slowest walker, total updates)."""
    import concurrent.futures as cf
    import multiprocessing as mp
    jobs = [(nbody, size, n_updates, 1000 + i) for i in range(cores)]
    t0 = time.perf_counter()
    with cf.ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn")) as ex:
        out = list(ex.map(_cpu_walker, jobs))
    wall = time.perf_counter() - t0
    return max(t for t, _ in out), sum(n for _, n in out), wall


def run_reference(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = max(1, a.ref_updates_per_step)
    times = []
    for i in range(a.warmup + a.steps):
        t, n, _ = cpu_walkers(a.nbody, a.stamp, per_step, cores)
        if i >= a.warmup:
            times.append(t)
    total_updates = per_step * cores * a.steps
    secs = sum(times)
    val = total_updates * a.stamp * a.stamp / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * secs / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "gibbs_updates_per_sec": total_updates / secs,
        "config": workload_config(a),
        "sample": "this arm runs a bounded SAMPLE of the workload: %d host walkers (one process per core) x %d "
                  "updates per step on epoch 0 of the same %dx%d stamps; the rate per update does not depend on "
                  "the number of walkers or epochs" % (cores, per_step, a.stamp, a.stamp),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d host walkers (one process each) x %d updates per step on epoch 0, "
                                   "%dx%d stamp, float64 numpy restatement of apf_step2.py:300-351 "
                                   "(the reference itself is Python 2 + astropy and cannot run here)"
                                   % (cores, per_step, a.stamp, a.stamp)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.path = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as fh:
            for ln in fh:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------
# GPU side
# ----------------------------------------------------------------------------------------------
def latency_block(a, dev):
    """BASELINE.json configs[0] and [1] -- one walker (apf_step2a) and 64 walkers (apf_step2 under
    mpiexec -n 64) on the 1024 x 1024 frame -- through the product path of the command lines:
    128-pixel stamp, whole-frame chi-square (the pixels outside the stamp through their sums), 16
    warps per walker.  Latency-bound by nature: reported beside the throughput line, not as it."""
    import torch
    from olpefit_b200 import frame, sampler, synth
    out = {}
    img, _ = synth.make_frame(0, a.nbody)
    size = 128
    ox, oy = synth.stamp_origin(size, a.nbody)
    guess = synth.step1_guess(img, a.nbody)
    p0 = frame.initial_parameters(img, guess, a.nbody)
    dom = frame.prepare_domain(torch.from_numpy(img).to(dev), HEADER, size=size, cut=(ox, oy), nbody=a.nbody,
                               device=str(dev), whole_frame=True)
    for name, walkers, n_upd in (("config1_one_walker", 1, 8192), ("config2_64_walkers", 64, 4096)):
        with sampler.GibbsSampler(dom, np.tile(p0, (walkers, 1)), seed=a.seed, burn_in=0, thin=16, team_warps=16) as s:
            s.run(256, record=False)                                  # warm-up
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = None
            for _ in range(3):
                e0.record()
                s.run(n_upd, record=False)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                best = ms if best is None else min(best, ms)
        out[name] = {"walkers": walkers, "stamp": size, "domain": "frame (1024 x 1024 through the outside sums)",
                     "team_warps": 16, "updates_per_launch": n_upd, "ms_per_launch": best,
                     "us_per_update_per_walker": 1e3 * best / n_upd,
                     "gibbs_updates_per_sec": walkers * n_upd / (best * 1e-3),
                     "pixel_model_evals_per_sec": walkers * n_upd * 1024.0 * 1024.0 / (best * 1e-3)}
    out["note"] = ("pixel_model_evals_per_sec counts the reference's domain (1024 x 1024 pixels per update); the Gaussians "
                   "are evaluated on the 128-pixel stamp, the rest of the frame enters through its exact sums")
    return out


def dump_outputs(out_dir, chain, seed):
    """Write chain rows [rows, walkers, P+1] to out_dir/chain.npy.  When they exceed DUMP_BYTES, a
    sample of walkers (drawn from ``seed``, kept in walker order) is written instead, the same
    walkers for the same arguments, so the dumps of two builds compare element for element."""
    import torch
    rows, walkers, cols = chain.shape
    keep = min(walkers, DUMP_BYTES // max(1, rows * cols * chain.element_size()))
    if keep < 1:
        raise SystemExit("--dump-outputs: the rows of one walker exceed %d bytes" % DUMP_BYTES)
    if keep < walkers:
        idx = np.sort(np.random.default_rng(seed).choice(walkers, keep, replace=False))
        chain = chain.index_select(1, torch.from_numpy(idx).to(chain.device))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "chain.npy"), chain.cpu().numpy())


def run_b200(a):
    cpu = None
    world_env = int(os.environ.get("WORLD_SIZE", 1))
    if world_env == 1 and not a.no_cpu_baseline:
        # before CUDA is touched in this process; rank 0 at N=1 only
        cores = os.cpu_count() or 1
        t, n, wall = cpu_walkers(a.nbody, a.stamp, a.cpu_updates, cores)
        sec_full = cpu_full_frame(a.nbody, 16)
        cpu = {"value": n * a.stamp * a.stamp / t, "unit": UNIT, "cores": cores, "kind": "port",
               "updates_per_sec": n / t, "seconds": round(wall, 2),
               "full_frame_1024": {"seconds_per_update_one_core": sec_full,
                                   "pixel_evals_per_sec_one_core": 1024 * 1024 / sec_full,
                                   "note": "the reference's own domain (whole frame per update), 1 core, 16 updates"},
               "sample": "%d host walkers (one process each, numpy float64 restatement of "
                         "apf_step2.py:300-351) x %d updates on epoch 0, %dx%d stamp"
                         % (cores, a.cpu_updates, a.stamp, a.stamp)}

    import ctypes as C
    import torch
    from olpefit_b200 import _lib, dist, frame, sampler, synth

    rank, local_rank, world = dist.init()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU path")
    if world > 1:
        # one slice of the host cores per rank: the ranks' Python threads and copy completions stop migrating
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, cores[local_rank * per:(local_rank + 1) * per] or cores)
        except (AttributeError, OSError):
            pass
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()

    W, F, S, U = a.walkers, a.frames, a.stamp, a.updates_per_step
    P = 3 * a.nbody + 10
    stamps, origins = synth.make_stamps(F, S, a.nbody)
    frame_of = (np.arange(W) % F).astype(np.int32)
    p_frame = []
    for f in range(F):
        g = synth.step1_guess(stamps[f], a.nbody, origin=tuple(origins[f]))
        p_frame.append(frame.initial_parameters(stamps[f], g, a.nbody, origin=tuple(origins[f])))
    init = np.asarray(p_frame)[frame_of]

    # pinned host copies: what a caller of the public API starts from
    frames_h = torch.from_numpy(stamps).pin_memory()
    init_h = torch.from_numpy(init).pin_memory()
    fo_h = torch.from_numpy(frame_of).pin_memory()

    def make_sampler(seed_offset=0):
        dom = frame.prepare_domain(frames_h.to(dev, non_blocking=True), HEADER, origin=origins, nbody=a.nbody)
        s = sampler.GibbsSampler(dom, init_h.to(dev, non_blocking=True), fo_h.to(dev, non_blocking=True),
                                 seed=a.seed + seed_offset, burn_in=0, thin=a.thin,
                                 id_base=rank * W, id_stride=1, team_warps=a.team)
        return dom, s

    dom, smp = make_sampler()
    rows = smp.rows_for(U)
    chain = torch.empty((max(rows, 1), W, P + 1), dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    for _ in range(a.warmup):
        smp.run(U, out=chain)
    torch.cuda.synchronize()
    dist.barrier()

    clocks = ClockSampler(local_rank) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    launches0 = smp.launches
    exps0 = int(smp.stats(moments=False)["exps"].item())
    launches0 = smp.launches
    torch.cuda.synchronize()
    dist.barrier()
    t_wall0 = time.perf_counter()
    for i in range(a.steps):
        flush.zero_()                       # evict stamps/state from L2 between timed steps
        ev[i][0].record()
        smp.run(U, out=chain)
        ev[i][1].record()
    torch.cuda.synchronize()
    dist.barrier()
    t_wall = time.perf_counter() - t_wall0
    gpu_launches = smp.launches - launches0
    ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
    ms = float(dist.allreduce_max(torch.tensor([ms], dtype=torch.float64, device=dev)).item())
    clk = clocks.stop() if clocks else None

    # cross-rank acceptance statistics (the only collective on this path), outside the timed region
    st = smp.stats(moments=False)
    tries, accepts, min_tries = dist.allreduce_stats(st["tries"], st["accepts"], st["min_tries"])
    exps_timed = float(dist.allreduce_sum((st["exps"] - exps0).double().reshape(1)).item())
    acc_rate = (accepts.double() / tries.double().clamp(min=1)).cpu().numpy()

    secs = ms * 1e-3
    updates = float(W) * U * a.steps * world
    value = updates * S * S / secs
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, chain[:rows], a.seed)

    # ---- end to end through the public API, host buffers in, host buffers out --------------
    # Every e2e step is a NEW batch of epochs: frames, starting points come from pinned host
    # memory, chain rows and counters go back to pinned host memory.  The sampler handle and
    # its device buffers are reused (lapf_sampler_reset), as a service processing a stream of
    # epochs would.
    e2e = None
    if not a.no_e2e:
        # chain rows leave the device as float32 differences from each walker's starting point
        # (LAPF_CHAIN_F32_DELTA: half the bytes, the values are restored exactly enough on the host)
        smp.set_chain_format("f32delta")
        chain32 = torch.empty((max(rows, 1), W, P + 1), dtype=torch.float32, device=dev)
        chain_h = torch.empty((max(rows, 1), W, P + 1), dtype=torch.float32).pin_memory()
        tot_h = torch.empty((2 * P + 1,), dtype=torch.int64).pin_memory()
        frames_d = torch.empty_like(frames_h, device=dev)
        init_d = torch.empty_like(init_h, device=dev)
        h2d = frames_h.numel() * 4 + init_h.numel() * 8
        d2h = chain_h.numel() * 4 + tot_h.numel() * 8
        n_e2e = max(3, a.steps)
        times = []
        names = ["h2d", "frame_prep", "reset_initial_chi2", "gibbs_updates", "d2h"]
        marks = [[torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)] for _ in range(n_e2e + 1)]
        host_ms = []
        for i in range(n_e2e + 1):
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            mk = marks[i]
            mk[0].record()
            frames_d.copy_(frames_h, non_blocking=True)
            init_d.copy_(init_h, non_blocking=True)
            mk[1].record()
            frame.prepare_domain(frames_d, HEADER, origin=origins, nbody=a.nbody, into=dom)
            mk[2].record()
            smp.reset(init_d, seed=a.seed + 1 + i)
            mk[3].record()
            ch = smp.run(U, out=chain32)
            mk[4].record()
            chain_h.copy_(ch, non_blocking=True)
            stt = smp.stats(moments=False)
            tot_h.copy_(torch.cat([stt["tries"], stt["accepts"], stt["min_tries"].reshape(1)]), non_blocking=True)
            mk[5].record()
            t_issue = time.perf_counter() - t0              # the host has queued the whole step
            torch.cuda.synchronize()
            dist.barrier()
            if i > 0:
                times.append(time.perf_counter() - t0)
                host_ms.append(1e3 * t_issue)
        phases = {nm: statistics.median(marks[i][j].elapsed_time(marks[i][j + 1]) for i in range(1, n_e2e + 1))
                  for j, nm in enumerate(names)}
        phases["host_issue"] = statistics.median(host_ms)
        if os.environ.get("LAPF_BENCH_DEBUG"):
            sys.stderr.write("e2e step times (ms): %s\n" % ["%.1f" % (1e3 * t) for t in times])
        # the same steps as a STREAM of epochs through the public double-buffered chain output
        # (sampler.ChainStreamer, K3): the chain rows of batch i travel to pinned host memory on the
        # copy stream while batch i+1 is uploaded, prepared and sampled.  Every copy of every step is
        # inside the timed region; the number is total wall time / steps.
        #
        # Two sampler handles (each with its pixel domain, chain streamer and compute stream) take the
        # batches in turn: upload, frame prep and initial chi-square of batch i+1 -- and the first
        # CTAs of its sampler kernel -- run while the last CTAs of batch i finish (the persistent kernel
        # holds every SM, so nothing of the NEXT batch can start on the same stream before it ends).
        dom_b, smp_b = make_sampler()
        smp_b.set_chain_format("f32delta")
        doms, smps = [dom, dom_b], [smp, smp_b]
        streamers = [sampler.ChainStreamer(smp, U), sampler.ChainStreamer(smp_b, U)]
        streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
        for st_ in streams:
            st_.wait_stream(torch.cuda.current_stream(dev))
        tot_hs = [torch.empty((2 * P + 1,), dtype=torch.int64).pin_memory() for _ in range(2)]
        got_rows = 0

        # the upload of a batch runs on its own stream into one of two buffer pairs, so it overlaps the
        # updates of the batch before (the host queues batch i+1 while batch i computes)
        up_stream = torch.cuda.Stream(device=dev)
        fr_d = [frames_d, torch.empty_like(frames_d)]
        in_d = [init_d, torch.empty_like(init_d)]
        uploaded = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def stream_step(i):
            j = i & 1
            compute, streamer = streams[j], streamers[j]
            up_stream.wait_event(consumed[j])              # the batch two steps ago has been read out of this pair
            with torch.cuda.stream(up_stream):
                fr_d[j].copy_(frames_h, non_blocking=True)
                in_d[j].copy_(init_h, non_blocking=True)
                uploaded[j].record(up_stream)
            with torch.cuda.stream(compute):
                compute.wait_event(uploaded[j])
                frame.prepare_domain(fr_d[j], HEADER, origin=origins, nbody=a.nbody, into=doms[j])
                smps[j].reset(in_d[j], seed=a.seed + 100 + i)
                consumed[j].record(compute)
                prev = streamer.run(U)
                stt = smps[j].stats(moments=False)
                tot_d = torch.cat([stt["tries"], stt["accepts"], stt["min_tries"].reshape(1)])
                # the counters leave on the copy stream too: a device->host copy queued on the compute stream would wait
                # behind the chain rows of this batch (one copy engine per direction) and hold up the next batch
                streamer.copy_stream.wait_stream(compute)
                with torch.cuda.stream(streamer.copy_stream):
                    tot_hs[j].copy_(tot_d, non_blocking=True)
                tot_d.record_stream(streamer.copy_stream)
            return 0 if prev is None else prev.shape[0]

        stream_step(0)                      # warm-up of both handles (allocations, first touch of the pinned buffers)
        stream_step(1)
        for sr in streamers:
            sr.finish()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        marks = [t0]
        for i in range(n_e2e):
            got_rows += stream_step(i + 2)
            marks.append(time.perf_counter())      # a batch has arrived in pinned host memory
        for sr in (streamers[n_e2e & 1], streamers[1 - (n_e2e & 1)]):       # the two batches still on their way, oldest first
            last = sr.finish()
            got_rows += 0 if last is None else last.shape[0]
        torch.cuda.synchronize()
        dist.barrier()
        t_total = (time.perf_counter() - t0) / n_e2e
        assert got_rows == rows * n_e2e, (got_rows, rows, n_e2e)
        # wall clock on a shared host is noisy (single steps of several 100 ms occur): the headline is
        # the MEDIAN interval between the arrivals of consecutive batches, the mean is reported too
        # (the first two timed steps hand nothing back -- each handle's first batch is still on its way)
        first = 3 if len(marks) > 6 else 1
        gaps = [b - a_ for a_, b in zip(marks[first:-1], marks[first + 1:])]
        if os.environ.get("LAPF_BENCH_DEBUG"):
            sys.stderr.write("e2e stream arrival gaps (ms): %s\n" % ["%.1f" % (1e3 * t) for t in gaps])
        t_stream = float(dist.allreduce_max(torch.tensor([statistics.median(gaps)], dtype=torch.float64, device=dev)).item())
        t_total = float(dist.allreduce_max(torch.tensor([t_total], dtype=torch.float64, device=dev)).item())
        # wall clock on a shared host is noisy: the headline uses the MEDIAN step (max over ranks);
        # mean, min and max are reported beside it
        t_med = float(dist.allreduce_max(torch.tensor([statistics.median(times)], dtype=torch.float64, device=dev)).item())
        t_mean = float(dist.allreduce_max(torch.tensor([sum(times) / len(times)], dtype=torch.float64, device=dev)).item())
        e2e = {"value": float(W) * U * world * S * S / t_stream, "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * t_stream, "ms_per_step_mean": 1e3 * t_total, "steps": n_e2e,
               "handles": 2,
               "what": "a stream of batches through the public API, taken in turn by two sampler handles on two "
                       "streams (the preparation of batch i+1 runs in the tail of batch i): per step pinned host frames + starting "
                       "points -> H2D (own stream, double-buffered) -> frame prep (mask, noise map) -> sampler reset (initial chi-square) -> "
                       "%d updates -> chain rows + counters D2H to pinned host, the chain rows double-buffered on "
                       "a copy stream (ChainStreamer) so they overlap the next batch; wall clock between the "
                       "arrivals of consecutive batches in host memory, median over steps (mean = total / steps "
                       "beside it), max over ranks" % U,
               "chain_rows": "float32 differences from the starting points (LAPF_CHAIN_F32_DELTA)",
               "phases_ms": dict({k: round(v, 3) for k, v in phases.items()},
                                 note="device time of each phase of one batch processed alone (CUDA events, median "
                                      "over steps, this rank) and the host time to queue the step; in the stream "
                                      "the d2h of batch i overlaps the phases of batch i+1"),
               "one_batch_at_a_time": {
                   "value": float(W) * U * world * S * S / t_med, "ms_per_step": 1e3 * t_med,
                   "ms_per_step_mean": 1e3 * t_mean, "ms_per_step_min": 1e3 * min(times),
                   "ms_per_step_max": 1e3 * max(times),
                   "what": "the same step with a device synchronisation on both sides (nothing overlaps); "
                           "wall clock per step, median over steps, max over ranks"}}

    smp.close()
    latency = latency_block(a, dev) if (rank == 0 and not a.no_latency) else None
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return

    # ---- roofline ---------------------------------------------------------------------------
    # SURVEY.md 8(d) counts per pixel-model evaluation K exponentials (SFU, its primary bound) and
    # 4K+3 FP32 instructions = 7K+4 flops (secondary bound).  The factorised kernel evaluates one
    # exponential per 4-pixel group instead of one per pixel, so the SFU no longer binds: the
    # kernel is bound by FP32 issue.  `achieved` is the survey's ALGORITHMIC flop count per
    # evaluation times the measured rate (it credits work the kernel avoids and may exceed what
    # the kernel really issues); `executed` is what the kernel really issues, from the device
    # counter of component evaluations left after far-field culling.
    pk = (C.c_double * 4)()
    _lib.check(lib.lapf_measure_peaks(pk))
    K = 2 * a.nbody
    NB = a.nbody
    per_gpu = value / world
    sm_count = int(pk[3])
    f_run = (clk or {}).get("sm_mhz") or pk[2]
    fp32_peak_flops = 2.0 * pk[1]                                   # measured FFMA stream, 2 flops per lane-FMA
    fp32_nominal = 2.0 * sm_count * 128 * f_run * 1e6
    alg_flops = per_gpu * (7 * K + 4)
    comp_rate = exps_timed / secs / world                           # component evaluations / s / GPU
    # lane operations the pixel loop issues per lane and warp step (8 pixels) for an active class:
    # 2 NB (anchor exponents) + 8 NB (C*E sums, packed) + 8 (block factor, packed) for 8 NB component
    # evaluations, i.e. (10 NB + 8) / (8 NB) each; per pixel 2 more (residual, square-accumulate)
    lane_ops = comp_rate * (10 * NB + 8) / (8.0 * NB) + per_gpu * 2.0
    ex2_alg = per_gpu * K
    # exponentials really issued: one per 2x4-pixel block and component + block/column tables per update
    upd_rate = per_gpu / (S * S)
    tr = min(S, 64)
    pw = min(S, 64)
    tab_ex2 = (S // 2) * 16 + (S // pw) * (S // tr) * (pw // 4) * K * 8
    ex2_exec = comp_rate / 8.0 + upd_rate * tab_ex2
    key = "%d-body %dx%d W=%d F=%d U=%d" % (a.nbody, S, S, W, F, U)
    traffic, ncu = None, None
    for name in ("r02_traffic.json", "r01_traffic.json"):          # per-launch DRAM bytes from the ncu --set full capture
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                tj = json.load(fh)
            if key in tj:
                traffic, ncu = tj[key], tj.get(key + " ncu")
                break
        except Exception:
            pass
    cyc_per_update = secs * f_run * 1e6 * sm_count * 4 / (updates / world)      # per scheduler (4 per SM)
    steps_per_update = (S // (4 if S >= 64 else 8)) * max(1, S // 64)
    exec_flops = 2.0 * lane_ops
    roofline = {
        "bound": "fp32", "kernel": ("gibbs_batch_kernel<%d,%d>" if a.team == 1 else "gibbs_kernel<%d,%d>") % (a.nbody, S),
        # the top-level numbers are what the silicon EXECUTES: FP32 lane operations of the pixel loop (FFMA = 2 flops)
        "achieved": exec_flops / 1e12, "peak": fp32_peak_flops / 1e12, "unit": "TFLOP/s",
        "frac": exec_flops / fp32_peak_flops,
        "what": "executed FP32 lane operations of the pixel loop ((10NB+8)/(8NB) per component evaluation left after "
                "far-field culling, from the device counter, + 2 per pixel) x 2 flops, against the measured FFMA-stream "
                "peak; tables, proposals and reductions are overhead and not counted",
        "peak_source": "measured on this device by lapf_measure_peaks (dependent-free FFMA stream x 2 flops); "
                       "MEASURED_PEAKS.json has no FP32 entry",
        "peak_nominal_at_run_clock": fp32_nominal / 1e12, "frac_nominal_at_run_clock": exec_flops / fp32_nominal,
        "executed": {
            "fp32_lane_ops_per_s": lane_ops, "fp32_lane_op_peak": pk[1], "frac": lane_ops / pk[1],
            "component_evals_per_pixel_eval": comp_rate / per_gpu,
            "ex2_per_s": ex2_exec, "ex2_per_pixel_eval": ex2_exec / per_gpu,
            "cycles_per_update_per_scheduler": cyc_per_update,
            "warp_steps_per_update": steps_per_update,
        },
        # the bound of the factorised loop, from tools/microbench7.cu on this GPU (profiles/r02_microbench7.txt):
        # a packed FFMA2 holds the FP32 pipe for 2 cycles, and for 3 when its three operand pairs all have to be
        # fetched from the register file; nothing else issues in its shadow
        "dispatch_model": {
            "fma_pipe_cycles_per_warp_step": 32 * 2 + 8,
            "operand_fetch_cycles_per_warp_step": 24 * 2.2 + 8 * 3.0 + 8 * 1.64,
            "other_instructions_per_warp_step": 17,
            "note": "2-body warp step (8 pixels x 4 components per lane): 32 packed + 8 scalar FP32 instructions + 4 "
                    "MUFU + 6 LDS.128 + 1 LDTM; measured costs: FFMA2 2.2 cycles with a reused operand, 3.0 with three "
                    "distinct pairs, FFMA 1.64 with distinct registers -> ~107 cycles per step per scheduler",
        },
        "ncu": ncu,                                                  # issue active, pipe utilisation of the committed capture
        "algorithmic": {
            "achieved": alg_flops / 1e12, "frac": alg_flops / fp32_peak_flops,
            "note": "SURVEY.md 8(d)'s count, %d flops (= %d FP32 instructions) and %d ex2 per pixel-model evaluation, x the "
                    "measured rate: credits work the factorised loop does not execute (not a utilisation)"
                    % (7 * K + 4, 4 * K + 3, K),
        },
        "sfu": {
            "achieved": ex2_alg / 1e9, "peak": pk[0] / 1e9, "unit": "Gex2/s", "frac": ex2_alg / pk[0],
            "frac_executed": ex2_exec / pk[0],
            "note": "the survey's primary bound: K ex2 per pixel-model evaluation against the measured MUFU.EX2 "
                    "peak; above 1 because the kernel issues %.2f ex2 per evaluation, not %d" % (ex2_exec / per_gpu, K),
        },
        "traffic": traffic,
    }
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "gibbs_updates_per_sec": updates / secs,
        "config": workload_config(a),
        "timing": {"how": "CUDA events around each step on the launch stream, summed; max over ranks",
                   "wall_ms_per_step_incl_flush": 1e3 * t_wall / a.steps},
        "clocks": clk, "e2e": e2e, "gpu_launches": int(gpu_launches),
        "roofline": roofline, "cpu_baseline": cpu, "latency": latency,
        "acceptance_rate_mean": float(np.mean(acc_rate)), "min_tries": int(min_tries.item()),
    }
    emit(line)


_JSON_FD = None


def emit(line):
    """The ONE JSON line goes to the process's original stdout; everything else that writes to
    file descriptor 1 (NCCL's version banner, library chatter) was redirected to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
