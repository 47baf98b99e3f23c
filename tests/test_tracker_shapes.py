"""The execution shapes of svob200_tracker_step and the frame store's level-0 binding.

A step runs as a CUDA graph with forked branches (device memory, batch <= 64), with the depth filter on its own stream
(device memory, larger batches), or in place on the context's stream (host-memory chunks of 256, profiling, chain mode).
These tests pin what each shape launches, that the profiling shape computes what the others compute, and that a frame
whose level 0 aliases a caller's device buffer takes its own storage back without touching that buffer."""
import ctypes as C
import numpy as np
import pytest

from android_svo_b200 import capi
from oracle import pyoracle_map as pm
import map_scenes as ms
import scenes
from test_pipeline import make_sequence

pytestmark = pytest.mark.gpu

ERR_ARG = -1                             # SVOB200_ERR_ARG
STAGES = ["frame+pyramid", "features_prepare", "sparse_align", "reproject_prepare", "match_geom", "match_prepare", "match_refine",
          "seeds_geom", "seeds_search", "seeds_refine", "seeds_finish", "stats"]


def c2_tracker(ctx, oracle, batch, mode, chain=False, n_frames=3, seed=0x00C0FFEE + 80):
    """A C2 tracker over `batch` sequences (3 distinct ones, replicated), its last frame set; returns it with a step function."""
    seqs = [make_sequence(oracle, "C2", seed + i, n_frames + 1) for i in range(min(batch, 3))]
    which = np.arange(batch) % len(seqs)
    cfg = seqs[0][0]
    N, S = cfg["n_features"], cfg["n_seeds"]
    trk = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), batch, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    take = lambda key: np.concatenate([seqs[w][3][key] for w in which])
    trk.set_keyframe(np.stack([seqs[w][2][0] for w in which]), np.stack([seqs[w][1][0] for w in which]), np.arange(batch + 1) * N,
                     take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S, take("seed_px"), take("seed_level"))
    if chain:
        trk.set_chain(30, 40, 1)
    (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in which]))

    def step(k):
        args = (np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                np.concatenate([seqs[w][4][k - 1] for w in which]))
        return (trk.step if mode == "host" else trk.step_device)(*args, want_px=True)
    return trk, step


# Kernel launches of one step, as ctx.launch_count() counts them (a graph replay counts the launches it was captured from).
# A default-mode step is 14 launches: pyramid 1, features_prepare + init_pose 2, sparse_align 1, points_select 1,
# match_direct 3 (geometry, prepare, refine), seed pose table 1, seeds_update 4 (geometry, search, refine, finish), step
# records 1.  The asynchronous depth filter writes the step records in two halves: 15.  A host-memory step of 300 sequences
# runs two chunks (256 + 44) of 14.  Chain mode replaces points_select and match_direct (4) with reproject_map (selection,
# match_direct's 3, cells: 5), chain_export, chain_segments and pose_optimize, and adds chain_stats: 19.
LAUNCHES = {("host", 3, False): 14, ("device", 3, False): 14, ("device", 70, False): 15, ("host", 300, False): 28,
            ("host", 3, True): 19, ("device", 3, True): 19}


def measure_launches(ctx, oracle):
    got = {}
    for mode, batch, chain in LAUNCHES:
        trk, step = c2_tracker(ctx, oracle, batch, mode, chain)
        try:
            per_step = []
            for k in (1, 2, 3):
                n0 = ctx.launch_count()
                step(k)
                per_step.append(ctx.launch_count() - n0)
            got[(mode, batch, chain)] = per_step
        finally:
            trk.close()
    return got


def test_launches_per_step(ctx, oracle):
    """Launches per step in each shape: graph replay (device, 3), asynchronous depth filter (device, 70), in place (host, 3),
    two host chunks (host, 300), and chain mode in host and device memory."""
    got = measure_launches(ctx, oracle)
    assert got == {key: [n] * 3 for key, n in LAUNCHES.items()}
    assert capi.load_library().svob200_tracker_launches_per_step() == 14


@pytest.mark.parametrize("batch", [3, 70])
def test_profiling_shape_computes_the_same(ctx, oracle, batch):
    """With stage profiling on, a device-memory step runs in place with direct launches between CUDA events (no graph, no
    depth-filter stream): its results are byte-identical to the same steps with profiling off, and every stage has a time."""
    out = {}
    for profiling in (False, True):
        trk, step = c2_tracker(ctx, oracle, batch, "device")
        try:
            trk.enable_profiling(profiling)
            rec = []
            for k in (1, 2, 3):
                stats, px, ok = step(k)
                rec.append((stats, px, ok, trk.seeds().copy(), trk.seed_obs().copy()))
                if profiling:
                    ms_ = trk.stage_ms()
                    assert list(ms_) == STAGES
                    assert all(np.isfinite(v) and v >= 0 for v in ms_.values()), ms_
            out[profiling] = rec
        finally:
            trk.close()
    for k, (a, b) in enumerate(zip(out[False], out[True])):
        for name, x, y in zip(("stats", "px", "ok", "seeds", "seed_obs"), a, b):
            assert x.tobytes() == y.tobytes(), "%s differs with profiling on at step %d" % (name, k + 1)
    assert out[False][-1][0]["n_matched"].min() > 20


def test_bind_then_take_back_own_storage(ctx, oracle):
    """A frame bound to a caller's device buffer (level 0 aliases it) takes its own storage back on every call that writes
    level 0 — frame_upload, frame_upload_level at level 0, frame_upload_yuv420 — and the caller's buffer stays as it was.  A
    bind with a misaligned pointer or stride is rejected and leaves level 0 where it was."""
    B, w, h, nl = 2, 160, 96, 3
    fid = 0x5A1D
    bound = np.stack([scenes.noise_image(h, w, 10 + b) for b in range(B)])
    d = ctx.dev_alloc(bound.nbytes)
    ctx.dev_upload(d, bound)
    ctx.frame_create(fid, B, w, h, nl)

    def check(imgs, what):
        for b in range(B):
            pyr = oracle.pyramid(imgs[b], nl)
            for l in range(nl):
                assert np.array_equal(ctx.frame_download(fid, b, l), pyr[l]), "%s: image %d level %d" % (what, b, l)
        back = np.zeros_like(bound)
        ctx.dev_download(back, d)
        assert np.array_equal(back, bound), "%s wrote into the caller's buffer" % what

    try:
        # host upload
        ctx.frame_bind(fid, d, w)
        check(bound, "bind")
        new = np.stack([scenes.noise_image(h, w, 20 + b) for b in range(B)])
        ctx.frame_upload(fid, new)
        check(new, "frame_upload")
        # every level of a host-side pyramid, level 0 first
        ctx.frame_bind(fid, d, w)
        new = np.stack([scenes.noise_image(h, w, 30 + b, blur=False) for b in range(B)])
        for b in range(B):
            for l, lv in enumerate(oracle.pyramid(new[b], nl)):
                lv = np.ascontiguousarray(lv)
                ctx._ck(ctx.L.svob200_frame_upload_level(ctx.h, fid, b, l, lv.ctypes.data_as(C.c_void_p), lv.shape[1]))
        check(new, "frame_upload_level")
        # YUV planes (planar chroma)
        ctx.frame_bind(fid, d, w)
        frames = [ms.yuv_frame(w, h, 40 + b, 1, 0) for b in range(B)]
        ybuf, ubuf, vbuf = (np.stack([fr[k] for fr in frames]) for k in ("y", "u", "v"))
        ctx.frame_upload_yuv420(fid, ybuf, ubuf, vbuf, frames[0]["y_stride"], frames[0]["uv_stride"], 1, ybuf[0].nbytes, ubuf[0].nbytes)
        om = pm.OracleMap(oracle)
        check(np.stack([om.yuv420_to_gray(fr["y"], fr["u"], fr["v"], fr["uv_stride"], 1, w, h, fr["y_stride"]) for fr in frames]), "frame_upload_yuv420")
        # rejected binds leave level 0 where it was: in the caller's buffer, then in the frame's own storage
        for before in (bound, new):
            if before is bound:
                ctx.frame_bind(fid, d, w)
            else:
                ctx.frame_upload(fid, new)
            for ptr, stride in ((d + 1, w), (d + 8, w), (d, w + 1), (d, w + 8), (d, w - 16)):
                rc = ctx.L.svob200_frame_bind(ctx.h, fid, C.c_void_p(ptr), stride, None)
                assert rc == ERR_ARG, (ptr - d, stride)
            for b in range(B):
                assert np.array_equal(ctx.frame_download(fid, b, 0), before[b])
    finally:
        ctx.frame_release(fid)
        ctx.dev_free(d)
