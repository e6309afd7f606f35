"""Drop-in command lines for step 2 of LAPF, driving the CUDA sampler.

    apf_step2.py IMAGE [-i {1,2a}]        apf_step2.py:154-158   (mpiexec -n N  ->  --walkers N)
    apf_step2a.py IMAGE                   apf_step2a.py:146-148
    3body/apf_step2_3body.py IMAGE        3body/apf_step2_3body.py:147-149

Same positional argument and -i flag, same step-1 input (<dir>/<N>_initialguess), same outputs
(<dir>/<N>_apf_results/<w>_finalarray_mpi.csv, <w>_acceptance_rate.csv, step2a.csv,
step2a_acceptance_rate), same defaults (accept_min = 100000; burn_in = 6000 / 0 for 3-body and
2a; n_steps = 5000).  New flags are additive.  Under torchrun the walkers are sharded over the
GPUs; every rank writes the files of its own walkers, so nothing but the stop rule and the
summary statistics crosses ranks.

Many epochs in one run (additive): ``--frames LIST`` names a text file with one FITS path per line.
Every frame keeps the reference's layout -- its own <N>_initialguess, its own <N>_apf_results/
with ``--walkers`` chains -- but all of them advance in ONE batched sampler, and the per-epoch
separation / position angle (median, 68 % interval, mean, std; apf_step3.py:283-291,436-437) and
Gelman-Rubin statistics (:260-278) are reduced on the device and written to
<N>_apf_results/step2_summary.json, so ``--no-chains`` runs need no chain to leave the GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np


def _positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError("must be a positive integer, got %s" % text)
    return v


def _parser(kind):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("image", type=str)
    if kind == "step2":
        ap.add_argument("-i", "--initial_guess_option", type=str,
                        help="Choose which file to take in as initial guess.  Enter -i 1 for step 1, "
                             "-i 2a for step 2a.")
    if kind != "step2a":
        ap.add_argument("--walkers", type=int, default=24,
                        help="independent walkers per image (replaces the process count of mpiexec -n)")
        ap.add_argument("--accept-min", type=int, default=100000,
                        help="stop when every parameter of every walker has been tried this often")
    else:
        ap.add_argument("--n-steps", type=int, default=5000)
    ap.add_argument("--frames", type=str, default=None,
                    help="text file with one FITS path per line: more epochs for the same run (each with its own "
                         "<N>_initialguess and <N>_apf_results/); IMAGE is the first epoch")
    ap.add_argument("--burn-in", type=int, default=None)
    ap.add_argument("--stamp", type=int, default=128, choices=[32, 64, 128],
                    help="side of the square cut-out, centred on the objects, in which the Gaussians are evaluated")
    ap.add_argument("--domain", choices=["frame", "stamp"], default="frame",
                    help="frame: chi-square over the whole image like the reference (pixels outside the stamp enter "
                         "through their exact sums against the constant floor); stamp: the cut-out only")
    ap.add_argument("--thin", type=int, default=1, help="record every thin-th update (1 = reference)")
    ap.add_argument("--seed", type=int, default=None, help="random seed (default: from the OS, like the reference's unseeded numpy)")
    ap.add_argument("--segment", type=int, default=4096, help="updates per kernel launch")
    ap.add_argument("--team", type=int, default=0, choices=[0, 1, 4, 16],
                    help="warps cooperating on one walker (0: pick from the total walker count)")
    ap.add_argument("--format", choices=["csv", "bin", "events"], default="csv",
                    help="per-walker reference CSV files, one packed binary, or (--thin 1 only) one packed file of "
                         "chain events: per update the parameter that was drawn, its value and chi-square, about a "
                         "seventh of the bytes of the rows; chains.read_packed / unpack_to_csv rebuild the rows")
    ap.add_argument("--chain-dtype", choices=["f64", "f32"], default="f64",
                    help="--format bin / events only: f32 stores float32 differences from each walker's starting point "
                         "(half the bytes off the device and on disk; chains.read_packed restores the values)")
    ap.add_argument("--no-chains", action="store_true",
                    help="record no chain rows at all: only the acceptance files and step2_summary.json (statistics "
                         "reduced on the device) are written")
    ap.add_argument("--fix-bkgd", action="store_true",
                    help="2-body only: use bkgd (p[9]) as the constant floor instead of the reference's p[12]")
    ap.add_argument("--adapt", action="store_true",
                    help="tune the jump widths from the acceptance rates DURING BURN-IN ONLY (the reference's widths "
                         "are fixed; off by default so posteriors compare like for like)")
    ap.add_argument("--checkpoint", action="store_true",
                    help="write <results>/checkpoint_rank<r>.pt when done (exact state of every walker)")
    ap.add_argument("--resume", action="store_true",
                    help="continue from <results>/checkpoint_rank<r>.pt, appending to the existing chain files "
                         "(give the --mcse / --ess-min, --draws and --adapt-per-epoch of the run that wrote it)")
    if kind != "step2a":
        ap.add_argument("--mcse", action="store_true",
                        help="keep batch means of every recorded value on the device: step2_summary.json gains the "
                             "effective sample size and Monte Carlo standard error of every parameter and of each "
                             "companion's separation and position angle")
        ap.add_argument("--ess-min", type=float, default=None,
                        help="(implies --mcse) stop once the separation and position-angle ESS of every companion "
                             "of every epoch is at least this; --accept-min stays the upper bound")
        ap.add_argument("--rhat-max", type=float, default=None,
                        help="stop once the Gelman-Rubin RC of every parameter of every epoch is at most this "
                             "(needs --walkers >= 2); with --ess-min both must hold")
        ap.add_argument("--draws", type=_positive_int, default=None, metavar="K",
                        help="keep a uniformly random sample of K recorded rows of every walker on the device and "
                             "write them to <results>/step2_draws.csv (also with --no-chains); step2_summary.json "
                             "gains the separation-PA correlation of these draws")
        ap.add_argument("--adapt-per-epoch", action="store_true",
                        help="give every epoch its own jump widths, tuned on the device DURING BURN-IN ONLY from that "
                             "epoch's acceptance in windows of at most %d updates (target %.2f); step2_summary.json "
                             "gains each epoch's widths and its acceptance after burn-in" % (ADAPT_WINDOW, ADAPT_TARGET))
    ap.add_argument("--quiet", action="store_true")
    return ap


MCSE_BATCH_ROWS, MCSE_LEVELS = 64, 16
# --adapt-per-epoch: windows [512 i, 512 (i + 1)) cut at the end of burn-in, and the acceptance they aim for
# (the constants of --adapt).  The windows are fixed in update counts, so a run resumed from a checkpoint
# adapts at the same counts as one that was never interrupted.
ADAPT_WINDOW, ADAPT_TARGET = 512, 0.35


def _burn_in(args, kind, nbody):
    if args.burn_in is not None:
        return args.burn_in
    return 6000 if (kind == "step2" and nbody == 2) else 0    # apf_step2.py:38; 3body :38; 2a: SURVEY C3


def _epoch_stats(sam, kind, nbody, n_frames, per_frame, n_local, world, bm_on):
    """Everything the summary and the stop rule read, reduced on the device and summed over ranks:
    Gelman-Rubin RC per epoch and parameter (apf_step3.py:260-278), the separation / position-angle
    sketch summary (:283-291,436-437) and the batch-means ESS / MCSE.  Every rank must call it."""
    import torch
    from . import chains, dist, stats
    out = {"rows": 0, "gelman_rubin": None, "sketch": None, "bm": None}
    P = sam.nparam
    stt = sam.stats(moments=True)
    n_rows = int(stt["rows"].item())
    out["rows"] = n_rows
    if kind != "step2a" and per_frame > 1 and n_rows > 1:
        mom = dist.allreduce_sum(stt["moments"] if n_local else torch.zeros_like(stt["moments"]))
        if world > 1:                     # the reference value of a frame is rank-local; all starts of a frame are equal here
            mom[:, :, 0] = mom[:, :, 0] / world
        mom = mom.cpu().numpy()
        out["gelman_rubin"] = [[float(v) for v in chains.gelman_rubin_from_moments(mom[f, :P], n_rows, per_frame)[1]]
                               for f in range(n_frames)]
    if kind != "step2a" and n_rows > 0:
        sk = sam.sketch()
        if not n_local:
            sk["hist"].zero_(); sk["summary"][..., 1:].zero_()
        sk["hist"] = dist.allreduce_sum(sk["hist"])
        sums = dist.allreduce_sum(sk["summary"][..., 1:].contiguous())
        sk["summary"] = torch.cat([sk["summary"][..., :1], sums], dim=-1)
        out["sketch"] = {k: v.cpu().numpy() for k, v in stats.sketch_summary(sk).items()}
    if bm_on and n_rows > 0:
        bm = sam.batch_means()
        bm["frame"] = dist.allreduce_sum(bm["frame"] if n_local else torch.zeros_like(bm["frame"]))
        res = stats.batch_means_summary(bm, torch.full((n_frames,), float(per_frame), dtype=torch.float64), n_rows)
        out["bm"] = {"ess": res["ess"].cpu().numpy(), "mcse": res["mcse"].cpu().numpy(),
                     "batch_rows": res["batch_rows_used"], "names": bm["names"]}
    return out


def _gather_draws(d, n_local, rank, world):
    """``GibbsSampler.draws()`` of every rank's first n_local walkers to rank 0 in global walker order
    (the interleaved sharding of dist.shard_ids): (values [W_total, K, P+1], rows [W_total, K]) as numpy
    arrays on rank 0, (None, None) elsewhere.  Every rank must call it."""
    from . import dist
    vals = d["values"][:n_local].transpose(0, 1).contiguous()                  # [K, W_local, P+1]
    rws = d["rows"][:n_local].transpose(0, 1).unsqueeze(-1).contiguous()     # [K, W_local, 1]
    parts_v, parts_r = dist.gather_chains(vals, rank, world), dist.gather_chains(rws, rank, world)
    if rank != 0:
        return None, None
    return (dist.merge_interleaved(parts_v).transpose(0, 1).cpu().numpy(),
            dist.merge_interleaved(parts_r)[..., 0].transpose(0, 1).cpu().numpy())


def _sep_pa_quantities(nbody):
    """Batch-mean quantities of the companions' separation and position angle (after the P+1 columns)."""
    p1 = 3 * nbody + 11
    return list(range(p1, p1 + 2 * (nbody - 1)))


def _converged(es, nbody, ess_min, rhat_max):
    """The stop rule on the output of _epoch_stats: every epoch meets every criterion given."""
    if ess_min is not None:
        bm = es["bm"]
        if bm is None or bm["batch_rows"] is None:
            return False
        ess = bm["ess"][:, _sep_pa_quantities(nbody)]
        if not (ess >= ess_min).all():          # nan (no level with enough batches yet) fails
            return False
    if rhat_max is not None:
        gr = es["gelman_rubin"]
        if gr is None or not (np.asarray(gr)[:, : 3 * nbody + 10] <= rhat_max).all():
            return False
    return True


def _frame_list(args):
    images = [args.image]
    if args.frames:
        base = os.path.dirname(os.path.abspath(args.frames))
        with open(args.frames) as fh:
            for ln in fh:
                ln = ln.strip()
                if not ln or ln.startswith("#"):
                    continue
                pth = ln if os.path.isabs(ln) else os.path.join(base, ln)
                if os.path.abspath(pth) not in [os.path.abspath(p) for p in images]:
                    images.append(pth)
    return images


def run(kind, nbody, argv=None):
    args = _parser(kind).parse_args(argv)
    if args.format == "events" and args.thin != 1:
        raise SystemExit("--format events needs --thin 1: rows further apart differ in more than one parameter")
    stop_rule = kind != "step2a" and (args.ess_min is not None or args.rhat_max is not None)
    bm_on = kind != "step2a" and (args.mcse or args.ess_min is not None)
    draws_k = getattr(args, "draws", None)
    if stop_rule and args.rhat_max is not None and args.walkers < 2:
        raise SystemExit("--rhat-max needs at least 2 walkers per epoch (Gelman-Rubin compares walkers)")
    burn_in = _burn_in(args, kind, nbody)
    adapt_pe = getattr(args, "adapt_per_epoch", False)
    if adapt_pe and args.adapt:
        raise SystemExit("--adapt-per-epoch and --adapt both tune the jump widths: give one of them")
    if adapt_pe and burn_in <= 0:
        raise SystemExit("--adapt-per-epoch tunes the widths during burn-in, and burn-in is 0: give --burn-in")
    import torch
    from . import chains, dist, frame, layout, sampler as smp, stats

    rank, local_rank, world = dist.init()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this implementation has no CPU path")
    torch.cuda.set_device(local_rank)
    device = "cuda:%d" % local_rank
    say = (lambda *a: None) if (args.quiet or rank != 0) else (lambda *a: print(*a, flush=True))

    images = _frame_list(args)
    n_frames = len(images)
    outdirs = [chains.results_dir(p) for p in images]
    say(outdirs[0] if n_frames == 1 else "%d epochs, results in %s ... %s" % (n_frames, outdirs[0], outdirs[-1]))
    if rank == 0:
        for d in outdirs:
            os.makedirs(d, exist_ok=True)                     # apf_step2.py:172-173
    dist.barrier()

    P = layout.nparam(nbody)
    from_2a = kind == "step2" and getattr(args, "initial_guess_option", None) == "2a"
    say("I am taking the initial guess from Step 2a output" if from_2a else "I am taking the initial guess from Step 1 output")

    def start_fn(image, hdr, path):
        if from_2a:                                                                # apf_step2.py:248-256
            a = np.genfromtxt(chains.results_dir(path) + "step2a.csv", delimiter=",")
            return np.array(a[-1][:P], dtype=np.float64)
        guess = np.loadtxt(open(chains.initial_guess_path(path), "rb"), delimiter=" ")   # :258-273
        return frame.initial_parameters(image, guess, nbody)

    floor_index = layout.bkgd_index(nbody) if (args.fix_bkgd and nbody == 2) else layout.REFERENCE_FLOOR_INDEX
    dom, params, cuts, headers = frame.load_epochs(images, start_fn, nbody=nbody, size=args.stamp,
                                                   floor_index=floor_index, device=device,
                                                   whole_frame=(args.domain == "frame"))
    if n_frames == 1:
        say("Masking pixels greater than ", 0.8 * frame.saturation_level(headers[0]))
    say("I have masked", int((dom.weight == 0).sum().item()), "pixels (inside the %dx%d domain%s)"
        % (args.stamp, args.stamp, " at x0=%d y0=%d" % tuple(cuts[0]) if n_frames == 1 else "s of all epochs"))

    per_frame = 1 if kind == "step2a" else args.walkers
    total_walkers = per_frame * n_frames
    id_base, id_stride, n_local = dist.shard_ids(total_walkers, rank, world)
    seed = args.seed if args.seed is not None else int.from_bytes(os.urandom(8), "little")
    if world > 1:   # every rank must use rank 0's seed
        t = torch.tensor([seed & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device=device)
        torch.distributed.broadcast(t, 0)
        seed = int(t.item())
    say("Random seed:", seed)
    if n_local == 0:
        say("rank has no walkers")
    # Few walkers: several warps per walker, so one update takes a fraction of the time; from about
    # 1,800 walkers per GPU the batched kernel (a warp owns 32 walkers) is faster (measured on B200:
    # 64 walkers 3.5e7 / 2.9e7 / 1.4e7 updates/s with 16 / 4 / 1 warps per walker, 592 walkers
    # 0.8e8 / 2.6e8 / 1.3e8, 2,048 walkers 0.8e8 / 2.2e8 / 2.4e8).  The choice depends on the TOTAL
    # walker count only, so every rank makes the same one.
    team = args.team
    if team == 0:
        team = 16 if (total_walkers <= 220 * world and args.stamp >= 64) else (4 if total_walkers <= 1800 * world else 1)
    # Global walker g = w * n_frames + frame: walker w of epoch `frame` (the reference's rank w of that image;
    # one epoch: g = w).  Ranks own g = rank (mod world), so with the epochs a multiple of the ranks every rank
    # owns WHOLE epochs (frame = rank mod world): its warps fill with walkers of one stamp (1,048 per
    # epoch instead of 131 at a million walkers, 1,000 epochs, 8 GPUs: +26 % at 32 pixels), and the
    # random streams -- keyed by g -- do not depend on the number of ranks.
    ids = np.array([id_base + i * id_stride for i in range(n_local)], dtype=np.int64)
    ids_or_0 = ids if n_local else np.zeros(1, dtype=np.int64)
    frame_of = (ids_or_0 % n_frames).astype(np.int32)
    sam = smp.GibbsSampler(dom, params[frame_of], frame_of, seed=seed, burn_in=burn_in,
                           thin=args.thin, id_base=id_base, id_stride=id_stride, team_warps=team)
    st0, _, _ = sam.state()
    if n_local:
        say("Found initial chi-squared:", float(st0[0, -1].item()))
        say("Initial guess:", np.concatenate([params[frame_of[0]], [float(st0[0, -1].item())]]))
    say()
    say("Beginning loop...")

    if kind == "step2a":
        paths = [outdirs[f] + "step2a.csv" for f in frame_of[:n_local]]
        acc_paths = [outdirs[f] + "step2a_acceptance_rate" for f in frame_of[:n_local]]
    else:
        paths = [outdirs[g % n_frames] + "%d_finalarray_mpi.csv" % (g // n_frames) for g in ids]
        acc_paths = [outdirs[g % n_frames] + "%d_acceptance_rate.csv" % (g // n_frames) for g in ids]

    # separation / position angle of every recorded row, binned on the device (one centre per epoch,
    # the same on every rank: the starting point)
    want_sketch = kind != "step2a"
    if want_sketch:
        centers = np.zeros((n_frames, nbody - 1, 2))
        for f in range(n_frames):
            for o in range(1, nbody):
                dx, dy = params[f][2 * o] - params[f][0], params[f][2 * o + 1] - params[f][1]
                centers[f, o - 1] = (np.hypot(dx, dy), np.degrees(np.arctan2(-dx, dy)))
        sam.enable_sketch(centers=centers)
    if bm_on:
        sam.enable_batch_means(MCSE_BATCH_ROWS, MCSE_LEVELS)
    if draws_k:
        sam.enable_draws(draws_k)
    if adapt_pe:
        sam.set_frame_widths()                # the default widths in every epoch's row, until burn-in tunes them

    def frame_counts():
        # per-epoch tries / accepts summed over ranks (a rank without walkers adds zeros); every rank must call it
        c = sam.frame_counts()
        return dist.allreduce_sum(c if n_local else torch.zeros_like(c))
    burn_counts = None                        # frame_counts() at the end of burn-in

    record = not args.no_chains
    f32 = args.format != "csv" and args.chain_dtype == "f32"
    # At --thin 1 consecutive rows differ in one parameter and chi-square: the rows leave the device as
    # events (a seventh of the bytes) and are rebuilt bit for bit on the host before the writers below.
    events = record and args.thin == 1
    if events:
        sam.set_chain_format("events_f32delta" if f32 else "events_f64")
    elif f32 and record:
        sam.set_chain_format("f32delta")
    packed = None
    if args.format != "csv" and record:
        packed = chains.PackedChainWriter(
            outdirs[0] + "chains_rank%d" % rank, max(n_local, 1), P + 1,
            {"walker_ids": ids.tolist(), "walkers_per_frame": per_frame, "frames": images, "seed": seed,
             "id_layout": "walker_id = walker * n_frames + frame",
             "burn_in": burn_in, "thin": args.thin, "nbody": nbody, "origin": [int(v) for v in cuts[0]],
             "cuts": cuts.tolist(), "stamp": args.stamp},
            dtype="float32" if f32 else "float64",
            start=sam.start().cpu().numpy() if f32 else None, resume=args.resume, events=args.format == "events")

    streamer = smp.ChainStreamer(sam, args.segment) if record else None
    first = [True]
    ckpt_path = outdirs[0] + "checkpoint_rank%d.pt" % rank
    if args.resume:
        ck = torch.load(ckpt_path)
        if ck["n_walkers"] != sam.n_walkers or ck["nbody"] != nbody:
            raise SystemExit("checkpoint %s does not match this run" % ckpt_path)
        sam.load(ck["blob"])
        seed = ck["seed"]
        if adapt_pe and ck.get("burn_counts") is not None:
            burn_counts = ck["burn_counts"].to(device)
        first[0] = False                      # append to the chain files that are already there
        say("Resumed at update", sam.count)
    widths, _is_log = layout.default_widths(nbody)

    def consume(seg):
        if seg is None or n_local == 0:
            return
        if args.format == "events":
            packed.append_events(*seg)
        else:
            if events:
                seg = chains.decode_events(*seg, sam.n_walkers, P + 1, np.float32 if f32 else np.float64)
            if packed is not None:
                packed.append(seg)
            else:
                chains.write_segment_csv(paths, seg, first[0])
        first[0] = False

    def advance(n):
        if record:
            consume(streamer.run(n))
        else:
            sam.run(n, record=False)

    stop = {"reason": "accept_min", "updates": 0}
    t_start = time.time()
    if kind == "step2a":
        left = args.n_steps                                   # apf_step2a.py:271
        while left > 0:
            n = min(args.segment, left)
            advance(n)
            left -= n
    else:
        while True:                                           # apf_step2.py:300
            stt = sam.stats(moments=False)
            tries, accepts, mn = dist.allreduce_stats(stt["tries"], stt["accepts"], stt["min_tries"])
            gap = args.accept_min - int(mn.item())
            if gap <= 0:
                break
            # min(tries) grows by at most one per update: `gap` updates can never overshoot
            n = min(args.segment, gap)
            if args.adapt and sam.count < burn_in:
                # burn-in only: nudge each width towards ~35% acceptance, then leave it alone
                n = min(n, max(burn_in - sam.count, 1), 512)
                if sam.count > 0:
                    rate = (accepts.double() / tries.double().clamp(min=1)).cpu().numpy()
                    widths = widths * np.clip(np.exp(rate - 0.35), 0.5, 2.0)
                    sam.set_widths(widths)
            if adapt_pe and sam.count < burn_in:
                n = min(n, burn_in - sam.count, ADAPT_WINDOW - sam.count % ADAPT_WINDOW)
            advance(n)
            if adapt_pe and sam.count <= burn_in and (sam.count % ADAPT_WINDOW == 0 or sam.count == burn_in):
                # the window that just ended lay in burn-in: every rank applies the same all-reduced counts
                counts = frame_counts()
                sam.adapt_widths(counts, ADAPT_TARGET)
                if sam.count == burn_in:
                    burn_counts = counts
            if sam.count % (10 * args.segment) < n:
                say("Loop count:", sam.count, " min tries:", int(mn.item()),
                    " acceptance rate:", (accepts.double() / tries.double().clamp(min=1)).cpu().numpy())
            if stop_rule and sam.count >= burn_in:
                # decided on rank 0 from all-reduced sums and broadcast: every rank stops at the same update
                es = _epoch_stats(sam, kind, nbody, n_frames, per_frame, n_local, world, bm_on)
                done = torch.tensor([1 if (rank == 0 and _converged(es, nbody, args.ess_min, args.rhat_max)) else 0],
                                    dtype=torch.int64, device=device)
                if world > 1:
                    torch.distributed.broadcast(done, 0)
                if int(done.item()):
                    stop["reason"] = "converged"
                    break
    if record:
        consume(streamer.finish())
    if packed is None and record and first[0] and n_local:
        for pth in paths:                                     # nothing recorded: the nan row alone
            chains.write_walker_csv(pth, np.zeros((0, P + 1)))
    if packed is not None:
        packed.close(count=sam.count)
    if args.adapt:
        say("Jump widths after burn-in tuning:", widths)
    if args.checkpoint and n_local:
        ck = {"blob": sam.save().cpu(), "n_walkers": sam.n_walkers, "nbody": nbody, "seed": seed, "count": sam.count}
        if adapt_pe:
            ck["burn_counts"] = None if burn_counts is None else burn_counts.cpu()
        torch.save(ck, ckpt_path)

    # Summary per epoch from statistics reduced on the device and summed over ranks -- no chain file
    # is read back: Gelman-Rubin per parameter (apf_step3.py:260-278), separation and position angle
    # of each companion (median, 68 % interval, mean, std; :283-291,436-437; without the distortion,
    # rotation and refraction corrections, whose tables are not part of the checkout).
    summaries = [dict(image=images[f], walkers=per_frame, updates=sam.count) for f in range(n_frames)]
    es = _epoch_stats(sam, kind, nbody, n_frames, per_frame, n_local, world, bm_on)
    n_rows = es["rows"]
    sep_pa_corr = {}                          # (epoch, companion - 1) -> correlation over the draws
    if draws_k:
        # every walker's reservoir to rank 0, in global walker order (g = w * n_frames + frame): the files
        # do not depend on the number of ranks
        all_v, all_r = _gather_draws(sam.draws(), n_local, rank, world)
        if rank == 0:
            col_names = list(layout.names(nbody)) + ["chi2"]
            for f in range(n_frames):
                v_f, r_f = all_v[f::n_frames], all_r[f::n_frames]
                count = chains.write_draws_csv(outdirs[f] + "step2_draws.csv", np.arange(per_frame), v_f, r_f, col_names)
                summaries[f]["draws"] = {"per_walker": draws_k, "rows_per_walker": n_rows, "count": count,
                                         "file": "step2_draws.csv"}
                pooled = torch.from_numpy(v_f[r_f >= 0])
                for o in range(1, nbody):
                    sep, pa = stats.separation_pa(pooled, companion=o)
                    corr = float(np.corrcoef(sep.numpy(), pa.numpy())[0, 1]) if count > 1 else float("nan")
                    sep_pa_corr[f, o - 1] = corr
    if es["gelman_rubin"] is not None:
        for f in range(n_frames):
            summaries[f]["gelman_rubin"] = es["gelman_rubin"][f]
        say("Gelman-Rubin stat per parameter (recorded rows, all walkers%s):" % ("" if n_frames == 1 else ", first epoch"),
            np.round(summaries[0]["gelman_rubin"], 4))
        say("GR for positions:", *np.round(summaries[0]["gelman_rubin"][:2 * nbody], 4))
    if want_sketch and n_rows > 0:
        res = es["sketch"]
        names = ["companion"] if nbody == 2 else ["b", "c"]
        for f in range(n_frames):
            for o, nm in enumerate(names):
                summaries[f]["sep_pa_%s" % nm] = {
                    "sep_mas": {"median": float(res["sep_q"][f, o, 1]), "lo": float(res["sep_q"][f, o, 0]),
                                "hi": float(res["sep_q"][f, o, 2]), "mean": float(res["sep_mean"][f, o]),
                                "std": float(res["sep_std"][f, o])},
                    "pa_deg": {"median": float(res["pa_q"][f, o, 1]), "lo": float(res["pa_q"][f, o, 0]),
                               "hi": float(res["pa_q"][f, o, 2]), "mean": float(res["pa_mean"][f, o]),
                               "std": float(res["pa_std"][f, o])},
                    "rows": int(res["count"][f, o]), "outside_histogram": float(res["outside"][f, o].max()),
                    "pixscale_mas": float(chains.PIXSCALE_PRE2015)}
                if (f, o) in sep_pa_corr:
                    # Pearson correlation of separation and position angle over the epoch's posterior draws
                    summaries[f]["sep_pa_%s" % nm]["sep_pa_corr"] = sep_pa_corr[f, o]
        if es["bm"] is not None:
            # Monte Carlo error of the means from the batch means (separation scaled to mas like the summary)
            bm = es["bm"]
            pnames = bm["names"][:P]
            for f in range(n_frames):
                summaries[f]["batch_rows"] = bm["batch_rows"]
                summaries[f]["ess"] = {nm: float(bm["ess"][f, j]) for j, nm in enumerate(pnames)}
                summaries[f]["mcse"] = {nm: float(bm["mcse"][f, j]) for j, nm in enumerate(pnames)}
                for o, nm in enumerate(names):
                    c = P + 1 + 2 * o
                    d = summaries[f]["sep_pa_%s" % nm]
                    d["sep_mas"]["ess"] = float(bm["ess"][f, c])
                    d["sep_mas"]["mcse"] = float(bm["mcse"][f, c] * chains.PIXSCALE_PRE2015)
                    d["pa_deg"]["ess"] = float(bm["ess"][f, c + 1])
                    d["pa_deg"]["mcse"] = float(bm["mcse"][f, c + 1])
        for f in range(min(n_frames, 8)):
            for nm in names:
                s_ = summaries[f]["sep_pa_%s" % nm]
                say("epoch %d %s: r = %.3f +%.3f -%.3f mas (std %.3f), pa = %.4f +%.4f -%.4f deg (std %.4f)  [%d rows]"
                    % (f, nm, s_["sep_mas"]["median"], s_["sep_mas"]["hi"] - s_["sep_mas"]["median"],
                       s_["sep_mas"]["median"] - s_["sep_mas"]["lo"], s_["sep_mas"]["std"], s_["pa_deg"]["median"],
                       s_["pa_deg"]["hi"] - s_["pa_deg"]["median"], s_["pa_deg"]["median"] - s_["pa_deg"]["lo"],
                       s_["pa_deg"]["std"], s_["rows"]))
                if "ess" in s_["sep_mas"]:
                    say("epoch %d %s: ESS r %.0f pa %.0f, MCSE r %.4f mas pa %.5f deg  [batches of %s rows]"
                        % (f, nm, s_["sep_mas"]["ess"], s_["pa_deg"]["ess"], s_["sep_mas"]["mcse"],
                           s_["pa_deg"]["mcse"], summaries[f]["batch_rows"]))
    if adapt_pe:
        # the widths every epoch ended burn-in with, and its acceptance over the updates after burn-in
        fw = sam.frame_widths().cpu().numpy()
        end = frame_counts().cpu().numpy()
        after = end - burn_counts.cpu().numpy() if burn_counts is not None else np.zeros_like(end)
        pnames = list(layout.names(nbody))
        for f in range(n_frames):
            summaries[f]["widths"] = {nm: float(fw[f, j]) for j, nm in enumerate(pnames)}
            summaries[f]["acceptance"] = {nm: (float(after[f, j, 1]) / float(after[f, j, 0]) if after[f, j, 0] > 0 else None)
                                          for j, nm in enumerate(pnames)}
        for f in range(min(n_frames, 8)):
            rate = after[f, :, 1] / np.maximum(after[f, :, 0], 1)
            say("epoch %d: acceptance after burn-in %s, jump widths %s"
                % (f, np.array2string(rate, precision=3), np.array2string(fw[f], precision=4)))
    if stop_rule or bm_on:
        stop["updates"] = sam.count
        for f in range(n_frames):
            summaries[f]["stop"] = dict(stop)
    if rank == 0 and kind != "step2a":
        for f in range(n_frames):
            with open(outdirs[f] + "step2_summary.json", "w") as fh:
                json.dump(summaries[f], fh, indent=1)
    _, tr, ac = sam.state()
    tr, ac = tr.cpu().numpy(), ac.cpu().numpy()
    for i in range(n_local):
        chains.write_acceptance(acc_paths[i], ac[i], tr[i])
    dist.barrier()
    say("Rank ", rank, "done with loop: %d updates per walker, %d walkers, %.1f s"
        % (sam.count, total_walkers, time.time() - t_start))
    sam.close()
    return 0


def main_step2(argv=None):
    return run("step2", 2, argv)


def main_step2a(argv=None):
    return run("step2a", 2, argv)


def main_step2_3body(argv=None):
    return run("step2_3body", 3, argv)


if __name__ == "__main__":
    sys.exit(main_step2())
