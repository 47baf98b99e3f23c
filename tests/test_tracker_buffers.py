"""Ownership of the tracker's device arrays.  They come in three groups, each made whole by the call that sizes it: the slots
(set_keyframe), the detector scratch (the first add_keyframes after set_keyframe or after set_detector changed the grid) and
the chain arrays (set_chain).  A group that is made again frees the one it replaces.  The sources are checked for the single
owner; svob200_tracker_device_bytes shows what the tracker holds across re-sizing; and a tracker that was re-sized computes
what a tracker sized once computes."""
import os
import re

import numpy as np
import pytest

from test_pipeline import gpu_step, make_sequence
from test_tracker_keyframes import add_keyframes_device, mask_of, tracker_state
from test_tracker_points import N_FRAMES, make_tracker
import scenes

TRACKER_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "android_svo_b200", "csrc", "tracker.cu")


# ---------------------------------------------------------------- the sources (no GPU)
def _tracker_src():
    return open(TRACKER_CU).read()


def test_one_owner_type_allocates():
    """Every device array of the tracker is allocated by the owner type's alloc (cudaMallocHost, the pinned staging, aside)."""
    src = _tracker_src()
    assert src.count("cudaMalloc(") == 1 and "class DevArrays {" in src
    owner = src[src.index("class DevArrays {"):]
    owner = owner[:owner.index("\n};\n")]
    assert "cudaMalloc(" in owner and "cudaFree(" in owner


def test_no_shared_owner_list_or_size_flag():
    src = _tracker_src()
    for word in ("alloc_owned", "owned", "det_cells_alloc"):
        assert not re.search(r"\b%s\b" % word, src), word


# ---------------------------------------------------------------- the device
@pytest.fixture(scope="module")
def seqs(oracle):
    return [make_sequence(oracle, "C2", 0x00C0FFEE + 60 + i, N_FRAMES + 1) for i in range(2)]


def step_args(seqs, data, k):
    """frame k of every sequence: images, the last poses and the map points' last pixels"""
    return (np.stack([seqs[w][2][k] for w in data]), np.stack([seqs[w][1][k - 1] for w in data]),
            np.concatenate([seqs[w][4][k - 1] for w in data]))


def insert(trk, mode, which, k):
    dm, dn = 2.0 + 0.01 * k, 1.0
    return trk.add_keyframes(which, dm, dn) if mode == "host" else add_keyframes_device(trk, which, dm, dn)


def plain_tracker(ctx, seqs, batch):
    """every seed of the keyframe, no seed or point pool (the trackers chain mode runs on)"""
    from android_svo_b200 import capi
    cfg = seqs[0][0]
    data = np.arange(batch) % 2
    N, S = cfg["n_features"], cfg["n_seeds"]
    trk = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), batch, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    take = lambda key: np.concatenate([seqs[w][3][key] for w in data])
    trk.set_keyframe(np.stack([seqs[w][2][0] for w in data]), np.stack([seqs[w][1][0] for w in data]), np.arange(batch + 1) * N,
                     take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S, take("seed_px"), take("seed_level"))
    return trk


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("batch", [3, 70])
def test_detector_scratch_is_replaced_not_added(ctx, seqs, mode, batch):
    """The first insertion adds the detector scratch once; steps and later insertions add nothing; a detector grid of another
    size gives the scratch back at once, and the next insertion makes it for the new grid: a finer grid holds more, and going
    back gives exactly the earlier total.  set_detector launches nothing."""
    data = np.arange(batch) % 2
    trk = make_tracker(ctx, seqs, batch, None, data)
    try:
        trk.set_detector(30, 3, 10.0)                          # before any insertion: nothing to give back
        base = trk.device_bytes()
        assert base > 0
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in data]))
        for k in range(1, 4):
            gpu_step(trk, mode, *step_args(seqs, data, k))
            assert trk.device_bytes() == base, "a step allocated (frame %d)" % k
        everyone = np.ones(batch, np.uint8)
        insert(trk, mode, everyone, 3)
        d30 = trk.device_bytes() - base
        assert d30 > 0
        gpu_step(trk, mode, *step_args(seqs, data, 4))
        insert(trk, mode, everyone, 4)
        gpu_step(trk, mode, *step_args(seqs, data, 5))
        assert trk.device_bytes() == base + d30
        n0 = ctx.launch_count()
        trk.set_detector(20, 3, 10.0)
        assert trk.device_bytes() == base and ctx.launch_count() == n0
        insert(trk, mode, everyone, 5)
        d20 = trk.device_bytes() - base
        assert d20 > d30
        gpu_step(trk, mode, *step_args(seqs, data, 6))
        n0 = ctx.launch_count()
        trk.set_detector(30, 3, 10.0)
        assert trk.device_bytes() == base and ctx.launch_count() == n0
        insert(trk, mode, everyone, 6)
        assert trk.device_bytes() == base + d30
    finally:
        trk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [3, 70])
def test_chain_arrays_are_replaced_not_added(ctx, seqs, batch):
    """set_chain(30), (20), (30): the first and the last total are equal, the finer grid holds more; set_chain(0) keeps the
    arrays for the next switch.  set_chain launches nothing."""
    trk = plain_tracker(ctx, seqs, batch)
    try:
        n0 = ctx.launch_count()
        trk.set_chain(30, 40, 1)
        b30 = trk.device_bytes()
        trk.set_chain(20, 40, 1)
        b20 = trk.device_bytes()
        trk.set_chain(30, 40, 1)
        assert trk.device_bytes() == b30 and b20 > b30
        trk.set_chain(0)
        assert trk.device_bytes() == b30
        assert ctx.launch_count() == n0
    finally:
        trk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch", [("device", 3), ("host", 70)])
def test_chain_resized_computes_the_same(ctx, seqs, mode, batch):
    """A tracker switched to chain cells 20, 30 and back to 20 steps byte for byte like one set to 20 once: step records,
    refined pixels, matches, seeds and seed observations."""
    data = np.arange(batch) % 2
    a, b = plain_tracker(ctx, seqs, batch), plain_tracker(ctx, seqs, batch)
    try:
        for cell in (20, 30, 20):
            a.set_chain(cell, 40, 1)
        b.set_chain(20, 40, 1)
        for t in (a, b):
            (t.set_last if mode == "host" else t.set_last_device)(np.stack([seqs[w][2][0] for w in data]))
        for k in range(1, 4):
            ra, rb = gpu_step(a, mode, *step_args(seqs, data, k), want_px=True), gpu_step(b, mode, *step_args(seqs, data, k), want_px=True)
            for name, x, y in zip(("stats", "px_refined", "match_ok"), ra, rb):
                assert x.tobytes() == y.tobytes(), "%s differs at frame %d" % (name, k)
            assert a.seeds().tobytes() == b.seeds().tobytes() and a.seed_obs().tobytes() == b.seed_obs().tobytes(), k
        assert ra[0]["n_matched"].min() > 20
    finally:
        a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch", [("host", 3), ("device", 70)])
def test_detector_resized_computes_the_same(ctx, seqs, mode, batch):
    """Tracker a makes its detector scratch for cell 20 (an insertion that selects nobody), then set_detector(30); tracker b is
    set to 30 from the start.  After the same steps and the same empty insertion, a staggered keyframe schedule leaves both in
    byte-identical states."""
    data = np.arange(batch) % 2
    a, b = make_tracker(ctx, seqs, batch, None, data), make_tracker(ctx, seqs, batch, None, data)
    try:
        b.set_detector(30, 3, 10.0)
        for t in (a, b):
            (t.set_last if mode == "host" else t.set_last_device)(np.stack([seqs[w][2][0] for w in data]))
            gpu_step(t, mode, *step_args(seqs, data, 1))
            insert(t, mode, np.zeros(batch, np.uint8), 1)
        a.set_detector(30, 3, 10.0)
        assert a.device_bytes() < b.device_bytes()                # a gave its scratch back
        n_kf = 0
        for k in range(2, N_FRAMES + 1):
            for t in (a, b):
                gpu_step(t, mode, *step_args(seqs, data, k))
            m = mask_of(batch, k)
            if m.any():
                na, nb = insert(a, mode, m, k), insert(b, mode, m, k)
                assert np.array_equal(na[0], nb[0]) and np.array_equal(na[1], nb[1]), k
                n_kf += int(m.sum())
            assert tracker_state(a) == tracker_state(b), "states differ after frame %d" % k
        assert n_kf > 0
        assert a.device_bytes() == b.device_bytes()
    finally:
        a.close(); b.close()
