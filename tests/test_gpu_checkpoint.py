"""Sampler checkpoints (lapf_sampler_save / lapf_sampler_load, include/lapf.h) for every combination of
sketches, batch means, draws and per-frame widths: the blob has the documented layout and holds what the
getters return; save / load continues the chains exactly; reset gives a new sampler's blob; and a blob
loads only into a sampler with the same batch means, draws and frame widths."""
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}
NBODY, SIZE, F, W, P = 2, 32, 2, 40, 16
MAX_PARAMS = 19                                   # LAPF_MAX_PARAMS
HEAD = 8 * (2 + MAX_PARAMS)
N_BINS, BM, K = 64, (3, 2), 5
SEED = 11
# (sketches, batch means, draws, frame widths)
COMBOS = list(itertools.product((False, True), repeat=4))


def _id(combo):
    return "-".join(n for n, on in zip(("sk", "bm", "dr", "fw"), combo) if on) or "plain"


@pytest.fixture(scope="module")
def gpu():
    import torch
    from olpefit_b200 import _lib, frame, layout, sampler, synth
    assert torch.cuda.is_available()
    stamps, origins = synth.make_stamps(F, SIZE, NBODY)
    dom = frame.prepare_domain(stamps, HEADER, origin=origins, nbody=NBODY)
    p_frame = np.array([synth.truth_parameters(NBODY, f) for f in range(F)])
    frame_of = np.arange(W) % F
    w0, _ = layout.default_widths(NBODY)
    return {"torch": torch, "lib": _lib, "sampler": sampler, "dom": dom, "init": p_frame[frame_of],
            "frame_of": frame_of, "table": np.stack([0.6 * w0, 1.9 * w0])}


def _sampler(gpu, combo, seed=SEED):
    sk, bm, dr, fw = combo
    s = gpu["sampler"].GibbsSampler(gpu["dom"], gpu["init"], gpu["frame_of"], seed=seed)
    if sk:
        s.enable_sketch(n_bins=N_BINS, sep_bin=1e-3, pa_bin=5e-3)
    if bm:
        s.enable_batch_means(*BM)
    if dr:
        s.enable_draws(K)
    if fw:
        s.set_frame_widths(gpu["table"])
    return s


def _advance(s, combo, a, b):
    """run(a), one adaptation step with frame widths, run(b); returns (the chains, the adaptation's counts)."""
    chains = [s.run(a).cpu().numpy()]
    counts = None
    if combo[3]:
        counts = s.frame_counts()
        s.adapt_widths(counts, 0.35)
        counts = counts.cpu().numpy()
    chains.append(s.run(b).cpu().numpy())
    return np.concatenate(chains), counts


def _layout(combo):
    """The table of include/lapf.h restated: ({part: (offset, bytes)}, [(offset, descriptor)], total bytes)."""
    sk, bm, dr, fw = combo
    slots = 2 * (NBODY - 1)
    C = P + 1 + (slots if sk else 0)
    sections = [(None, [("state", 8 * W * (P + 1)), ("shift", 8 * W * (P + 1)), ("moments", 16 * W * (P + 1)),
                        ("exps", 8 * W), ("tries", 4 * W * P), ("accepts", 4 * W * P)])]
    if sk:
        sections.append((None, [("sk_mom", 8 * W * slots * 2), ("sk_hist", 4 * F * slots * (N_BINS + 2))]))
    if bm:
        sections.append(((b"LAPFBM01", BM[0], BM[1], C), [("bm", 8 * W * C * BM[1] * 2)]))
    if dr:
        sections.append(((b"LAPFRS01", K, P + 1, 0), [("dr_val", 8 * W * K * (P + 1)), ("dr_row", 8 * W * K)]))
    if fw:
        sections.append(((b"LAPFFW01", F, P, 0), [("fw", 8 * F * P), ("fw_snap", 16 * F * P)]))
    off, parts, descs = HEAD, {}, []
    for desc, ps in sections:
        if desc:
            descs.append((off, desc))
            off += 32
        for name, nb in ps:
            parts[name] = (off, nb)
            off += nb
    return parts, descs, off


def _same_bytes(a, b, msg=""):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    np.testing.assert_array_equal(a.reshape(-1).view(np.uint8), b.reshape(-1).view(np.uint8), err_msg=msg)


def _observe(s, combo):
    """Everything the getters report, as numpy."""
    sk, bm, dr, fw = combo
    st, tr, ac = (t.cpu().numpy() for t in s.state())
    out = {"state": st, "tries": tr, "accepts": ac, "start": s.start().cpu().numpy(),
           "moments": s.stats()["moments"].cpu().numpy(), "counts": s.frame_counts().cpu().numpy()}
    if sk:
        k = s.sketch()
        out["hist"], out["summary"] = k["hist"].cpu().numpy(), k["summary"].cpu().numpy()
    if bm:
        m = s.batch_means()
        out["bm_walker"], out["bm_frame"] = m["walker"].cpu().numpy(), m["frame"].cpu().numpy()
    if dr:
        d = s.draws()
        out["draws"], out["draw_rows"] = d["values"].cpu().numpy(), d["rows"].cpu().numpy()
    if fw:
        out["fw"] = s.frame_widths().cpu().numpy()
    return out


@pytest.mark.parametrize("combo", COMBOS, ids=_id)
def test_blob_has_the_documented_layout_and_the_getters_values(gpu, combo):
    sk, bm, dr, fw = combo
    with _sampler(gpu, combo) as s:
        _, counts = _advance(s, combo, 37, 20)
        blob = s.save().cpu().numpy()
        parts, descs, total = _layout(combo)
        assert blob.size == total
        head = blob[:HEAD].view(np.int64)
        assert head[0] == 57 and head[1] == SEED
        for off, desc in descs:
            assert bytes(blob[off:off + 8]) == desc[0]
            assert blob[off + 8:off + 32].view(np.int64).tolist() == list(desc[1:])

        def region(name):
            off, nb = parts[name]
            return blob[off:off + nb]

        got = _observe(s, combo)
        for name, key in (("state", "state"), ("tries", "tries"), ("accepts", "accepts"), ("shift", "start")):
            _same_bytes(region(name), got[key], name)
        if sk:
            np.testing.assert_array_equal(region("sk_hist").view(np.uint32), got["hist"].reshape(-1))
        if bm:
            _same_bytes(region("bm"), got["bm_walker"])
        if dr:
            _same_bytes(region("dr_val"), got["draws"])
            _same_bytes(region("dr_row"), got["draw_rows"])
        if fw:
            _same_bytes(region("fw"), got["fw"])
            assert not np.array_equal(got["fw"], gpu["table"])         # the adaptation step changed the widths
            _same_bytes(region("fw_snap"), counts)                    # ... and left its counts as the snapshot
            assert counts.any()


@pytest.mark.parametrize("combo", COMBOS, ids=_id)
def test_save_load_continues_the_chains_exactly(gpu, combo):
    with _sampler(gpu, combo) as s:
        _advance(s, combo, 30, 9)
        blob = s.save().clone()
        chains_a, _ = _advance(s, combo, 17, 12)
        got_a, blob_a = _observe(s, combo), s.save().cpu().numpy()
        s.load(blob)
        chains_b, _ = _advance(s, combo, 17, 12)
        got_b, blob_b = _observe(s, combo), s.save().cpu().numpy()
    _same_bytes(chains_a, chains_b, "chains")
    for key in got_a:
        _same_bytes(got_a[key], got_b[key], key)
    _same_bytes(blob_a, blob_b, "blob")


@pytest.mark.parametrize("combo", COMBOS, ids=_id)
def test_reset_gives_a_new_samplers_blob(gpu, combo):
    with _sampler(gpu, combo) as s:
        _advance(s, combo, 41, 13)
        s.reset(gpu["init"], seed=23)
        if combo[3]:
            s.set_frame_widths(gpu["table"])
        got = s.save().cpu().numpy()
    with _sampler(gpu, combo, seed=23) as t:
        want = t.save().cpu().numpy()
    _same_bytes(got, want)


@pytest.mark.parametrize("sketch", [False, True], ids=["plain", "sk"])
def test_blob_loads_only_into_the_same_optional_state(gpu, sketch):
    torch, lib = gpu["torch"], gpu["lib"]
    combos = [c for c in COMBOS if c[0] == sketch]
    blobs = {}
    for c in combos:
        with _sampler(gpu, c) as s:
            _advance(s, c, 21, 8)
            blobs[c] = s.save().clone()
    for b in combos:
        with _sampler(gpu, b, seed=5) as t:
            t.run(3)
            before = t.save().clone()
            for a in combos:
                if a != b:
                    with pytest.raises(lib.LapfError):
                        t.load(blobs[a])
                    assert torch.equal(t.save(), before), (_id(a), _id(b))
            t.load(blobs[b])
            assert torch.equal(t.save(), blobs[b])
    # the refusals name the sections involved
    plain, bm, dr = (sketch, False, False, False), (sketch, True, False, False), (sketch, False, True, False)
    with _sampler(gpu, plain) as t:
        with pytest.raises(lib.LapfError, match="carries batch means, this sampler has none"):
            t.load(blobs[bm])
    with _sampler(gpu, bm) as t:
        with pytest.raises(lib.LapfError, match="carries posterior draws where this sampler expects batch means"):
            t.load(blobs[dr])
