"""Per-sequence keyframes (svob200_tracker_add_keyframes, svob200_tracker_scene_depth): every sequence of the batch takes its
keyframes on its own frames, in its own ring, like one FrameHandlerMono + DepthFilter per sequence.  All-ones masks against
svob200_tracker_add_keyframe, staggered schedules against one oracle per schedule, the scene depth against a CPU restatement,
a device-only keyframe loop against the same schedule in host memory, and the argument checks."""
import ctypes as C

import numpy as np
import pytest

from oracle.pyoracle import Cam, OracleSeq
from test_pipeline import KF_DET, gpu_step, make_sequence, seed_matrix
from test_tracker_points import CAP_BIG, POOL, S0, N_FRAMES, bits, depth_args, last_px_of, make_tracker, oracle_seq
import scenes

CAP = 2400                                   # seed slots per sequence (make_tracker)


@pytest.fixture(scope="module")
def seqs(oracle):
    return [make_sequence(oracle, "C2", 0x00C0FFEE + 60 + i, N_FRAMES + 1) for i in range(2)]


def schedule(c, k):
    """does a sequence of schedule class c take a keyframe after frame k?  Class 3 never does; the others fill and evict
    their rings at different frames."""
    return (k % 2 == 0, k % 3 == 1, k in (4, 5, 9, 10, 11), False)[c]


def mask_of(batch, k):
    return np.array([schedule(b % 4, k) for b in range(batch)], np.uint8)


def dev_array(ctx, a):
    p = ctx.dev_alloc(max(a.nbytes, 8))
    ctx.dev_upload(p, a)
    return p


def add_keyframes_device(trk, which, dm, dn):
    """add_keyframes with every array in device memory; returns the counts read back"""
    ctx, B = trk.ctx, trk.batch
    dm = np.ascontiguousarray(np.broadcast_to(np.asarray(dm, np.float32), (B,)))
    dn = np.ascontiguousarray(np.broadcast_to(np.asarray(dn, np.float32), (B,)))
    ptrs = [dev_array(ctx, a) for a in (np.asarray(which, np.uint8) if which is not None else np.zeros(1, np.uint8), dm, dn,
                                        np.full(B, -5, np.int32), np.full(B, -5, np.int32))]
    try:
        trk.add_keyframes_raw(ptrs[0] if which is not None else 0, ptrs[1], ptrs[2], ptrs[3], ptrs[4])
        ctx.sync()
        n_new, n_drop = np.zeros(B, np.int32), np.zeros(B, np.int32)
        ctx.dev_download(n_new, ptrs[3]); ctx.dev_download(n_drop, ptrs[4])
    finally:
        for p in ptrs:
            ctx.dev_free(p)
    return n_new, n_drop


def tracker_state(trk):
    pos, ty, no, cr, dr = trk.points()
    return dict(seeds=trk.seeds().tobytes(), refs=[np.asarray(x).tobytes() for x in trk.seed_refs()], obs=trk.seed_obs().tobytes(),
                pos=bits(pos).tobytes(), ty=ty.tobytes(), no=no.tobytes(), cr=cr.tobytes(), dr=dr.tobytes())


# ---------------------------------------------------------------- 1. all-ones masks = add_keyframe
@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch", [("device", 3), ("device", 70), ("host", 300)])
def test_all_ones_equals_add_keyframe(ctx, oracle, seqs, mode, batch):
    """Two trackers on the same inputs, one inserting with add_keyframe, the other with add_keyframes (which = NULL, an all-ones
    host mask, an all-ones mask in device memory, in turn): byte-identical step records, matches, seeds, seed references, seed
    observations and point slots after every step and keyframe.  B = 3 replays graphs, B = 70 runs the asynchronous depth
    filter, B = 300 steps in two host-memory chunks.  add_keyframe is add_keyframes for every sequence in host memory, so this
    compares the three ways of selecting every sequence with each other; that add_keyframe computes what it computed before
    rests on the oracle comparisons of tests/test_pipeline.py::test_tracker_keyframe_insertion_matches_oracle and
    tests/test_tracker_points.py, which are unchanged."""
    cfg = seqs[0][0]
    which = np.arange(batch) % 2
    a, b = make_tracker(ctx, seqs, batch, CAP_BIG, which), make_tracker(ctx, seqs, batch, CAP_BIG, which)
    try:
        for t in (a, b):
            (t.set_last if mode == "host" else t.set_last_device)(np.stack([seqs[w][2][0] for w in which]))
        n_kf = 0
        for k in range(1, N_FRAMES + 1):
            pos, ty = a.points()[:2]
            lp = np.concatenate([last_px_of(cfg, seqs[w][1][k - 1], pos[i * CAP_BIG:(i + 1) * CAP_BIG], ty[i * CAP_BIG:(i + 1) * CAP_BIG])
                                 for i, w in enumerate(which)])
            args = (np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]), lp)
            ra, rb = gpu_step(a, mode, *args, want_px=True), gpu_step(b, mode, *args, want_px=True)
            assert ra[0].tobytes() == rb[0].tobytes() and bits(ra[1]).tobytes() == bits(rb[1]).tobytes() and ra[2].tobytes() == rb[2].tobytes(), k
            assert tracker_state(a) == tracker_state(b), "state differs after frame %d" % k
            if k % 3 == 0:
                na = a.add_keyframe(*depth_args(k))
                variant = n_kf % 3
                if variant == 0:
                    nb = b.add_keyframes(None, *depth_args(k))
                elif variant == 1:
                    nb = b.add_keyframes(np.ones(batch, np.uint8), *depth_args(k))
                else:
                    nb = add_keyframes_device(b, np.ones(batch, np.uint8), *depth_args(k))
                n_kf += 1
                assert np.array_equal(na[0], nb[0]) and np.array_equal(na[1], nb[1]), "counts differ at keyframe %d" % k
                assert na[0].min() > 0
                assert tracker_state(a) == tracker_state(b), "state differs after keyframe %d (variant %d)" % (k, variant)
        assert n_kf == 4
    finally:
        a.close(); b.close()


# ---------------------------------------------------------------- 2. staggered schedules against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("batch", [2, 70])
def test_staggered_keyframes_match_oracle(ctx, oracle, seqs, batch, mode):
    """Sequence b follows schedule class b % 4 (its data: b % 2), one pinned oracle per class that calls add_keyframe on that
    class's frames only: new-seed counts (0 where not selected), pool occupancy slot by slot, keyframe indices and batch ids,
    seed statuses and seed bits under the device's pose, closest-view map-point matches."""
    from android_svo_b200 import capi
    n_cls = min(batch, 4)
    cfg = seqs[0][0]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    N = cfg["n_features"]
    data = np.arange(batch) % 2
    cls = np.arange(batch) % 4
    pinned = [OracleSeq(oracle, cam_o, *args, 100.0, 2.4, 1.2, POOL[2]) for _ in range(n_cls)]
    trk = capi.Tracker(ctx, cam_g, batch, *args)
    try:
        trk.set_seed_pool(CAP, *POOL); trk.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
        for c, s in enumerate(pinned):
            _, poses, imgs, kf, _ = seqs[c % 2]
            s.set_pool(*POOL); s.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"][:S0], kf["seed_level"][:S0])
            s.set_last(imgs[0])
        take = lambda key, n=None: np.concatenate([seqs[w][3][key][:n] for w in data])
        trk.set_keyframe(np.stack([seqs[w][2][0] for w in data]), np.stack([seqs[w][1][0] for w in data]), np.arange(batch + 1) * N,
                         take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S0, take("seed_px", S0), take("seed_level", S0))
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in data]))
        n_bit_diff = n_seedframes = 0
        for k in range(1, N_FRAMES + 1):
            stats, px_g, ok_g = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in data]), np.stack([seqs[w][1][k - 1] for w in data]),
                                         np.concatenate([seqs[w][4][k - 1] for w in data]), want_px=True)
            for c in range(n_cls):
                pinned[c].set_pose_override(stats[c]["T_cur_w"])
                _, px_o, ok_o = pinned[c].step(seqs[c % 2][2][k], seqs[c % 2][1][k - 1], seqs[c % 2][4][k - 1], want_px=True)
                for b in np.nonzero(cls == c)[0][:3]:
                    assert np.array_equal(ok_g[b * N:(b + 1) * N], ok_o) and np.array_equal(px_g[b * N:(b + 1) * N], px_o), \
                        "map-point matches differ (seq %d, frame %d)" % (b, k)
            m = mask_of(batch, k)
            if m.any():
                dm, dn = depth_args(k)
                n_new, n_drop = (trk.add_keyframes(m, dm, dn) if mode == "host" else add_keyframes_device(trk, m, dm, dn))
                assert (n_new[m == 0] == 0).all() and (n_drop == 0).all()
                for c in range(n_cls):
                    if schedule(c, k):
                        n_o = pinned[c].add_keyframe(dm, dn)
                        assert (n_new[cls == c] == n_o).all(), "new-seed count differs at frame %d: %s vs %d" % (k, n_new[cls == c][:4], n_o)
            px, lv, kfi, bt, st = trk.seed_refs()
            seeds_g, obs_g = seed_matrix(trk.seeds()), trk.seed_obs()
            for b in range(batch):
                c = cls[b]
                opx, olv, okf, obt, ost = pinned[c].seed_refs()
                So = len(olv)
                sl = slice(b * CAP, b * CAP + So)
                assert np.array_equal(st[sl], ost) and (st[b * CAP + So:(b + 1) * CAP] == 1).all(), "pool occupancy differs (seq %d, frame %d)" % (b, k)
                alive = ost == 0
                assert np.array_equal(px[sl][alive], opx[alive]) and np.array_equal(lv[sl][alive], olv[alive])
                assert np.array_equal(kfi[sl][alive], okf[alive]) and np.array_equal(bt[sl][alive], obt[alive]), "kf / batch ids differ (seq %d, frame %d)" % (b, k)
                n_bit_diff += int((seeds_g[sl][alive].view(np.uint32) != pinned[c].seeds()[alive].view(np.uint32)).any(axis=1).sum())
                n_seedframes += int(alive.sum())
                assert np.array_equal(obs_g["status"][sl], pinned[c].seed_obs()["status"]), "seed statuses differ (seq %d, frame %d)" % (b, k)
        print("staggered keyframes: %d seed-frames, %d bit differences under the device's pose" % (n_seedframes, n_bit_diff))
        assert n_bit_diff == 0
        # the rings evicted at different frames: at the end every keyframing class holds seeds of several keyframes, the
        # class that never takes one only seeds of its first keyframe
        for b in range(min(batch, 4)):
            alive = st[b * CAP:(b + 1) * CAP] == 0
            assert (len(np.unique(kfi[b * CAP:(b + 1) * CAP][alive])) >= 2) == (cls[b] != 3)
    finally:
        trk.close()
        for s in pinned:
            s.close()


# ---------------------------------------------------------------- 3. staggered schedules with a point pool
@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch", [("host", 4), ("device", 70)])
def test_staggered_keyframes_point_pool_match_oracle(ctx, oracle, seqs, mode, batch):
    """The point pool under per-sequence schedules against one PoolSeq per schedule class: positions bit for bit, types,
    observation counts, created / dropped, matches and refined pixels, seed states and statuses."""
    n_cls = min(batch, 4)
    cfg = seqs[0][0]
    data = np.arange(batch) % 2
    cls = np.arange(batch) % 4
    pinned = [oracle_seq(seqs[c % 2], CAP_BIG) for c in range(n_cls)]
    trk = make_tracker(ctx, seqs, batch, CAP_BIG, data)
    P = CAP_BIG
    try:
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in data]))
        promoted = evicted = 0

        def compare(k, what):
            pos, ty, no, cr, dr = trk.points()
            seeds_g = seed_matrix(trk.seeds())
            obs_g = trk.seed_obs()
            _, _, _, _, st = trk.seed_refs()
            for b in range(batch):
                c = cls[b]
                opos, oty, ono, ocr, odr = pinned[c].points()
                sl = slice(b * P, (b + 1) * P)
                assert np.array_equal(bits(pos[sl]), bits(opos)), "positions differ (seq %d, %s %d)" % (b, what, k)
                assert np.array_equal(ty[sl], oty) and np.array_equal(no[sl], ono), "types / observations differ (seq %d, %s %d)" % (b, what, k)
                assert (cr[b], dr[b]) == (ocr, odr), "created / dropped differ (seq %d, %s %d)" % (b, what, k)
                So = pinned[c].num_slots()
                ssl = slice(b * CAP, b * CAP + So)
                ost = pinned[c].seed_refs()[4]
                assert np.array_equal(st[ssl], ost)
                alive = ost == 0
                assert np.array_equal(seeds_g[ssl][alive].view(np.uint32), pinned[c].seeds()[alive].view(np.uint32)), "seeds differ (seq %d, %s %d)" % (b, what, k)
                assert np.array_equal(obs_g["status"][ssl], pinned[c].seed_obs()["status"])
            return ty

        ty_prev = trk.points()[1]
        for k in range(1, N_FRAMES + 1):
            lp = [last_px_of(cfg, seqs[c % 2][1][k - 1], *pinned[c].points()[:2]) for c in range(n_cls)]
            stats, px_g, ok_g = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in data]), np.stack([seqs[w][1][k - 1] for w in data]),
                                         np.concatenate([lp[c] for c in cls]), want_px=True)
            for c in range(n_cls):
                pinned[c].set_pose_override(stats[c]["T_cur_w"])
                _, px_o, ok_o = pinned[c].step(seqs[c % 2][2][k], seqs[c % 2][1][k - 1], lp[c], want_px=True)
                for b in np.nonzero(cls == c)[0]:
                    assert np.array_equal(ok_g[b * P:(b + 1) * P], ok_o) and np.array_equal(bits(px_g[b * P:(b + 1) * P]), bits(px_o)), \
                        "matches differ (seq %d, frame %d)" % (b, k)
            ty_prev = compare(k, "frame")
            m = mask_of(batch, k)
            if m.any():
                dm, dn = depth_args(k)
                n_new, _ = trk.add_keyframes(m, dm, dn) if mode == "host" else add_keyframes_device(trk, m, dm, dn)
                for c in range(n_cls):
                    if schedule(c, k):
                        assert (n_new[cls == c] == pinned[c].add_keyframe(dm, dn)).all()
                ty = compare(k, "keyframe")
                promoted += int(((ty_prev == 1) & (ty == 2)).sum())
                evicted += int(((ty_prev == 1) & (ty == 0)).sum())
        print("staggered point pool: promoted %d, deleted by eviction %d" % (promoted, evicted))
        assert promoted > 0 and evicted > 0
    finally:
        trk.close()
        for s in pinned:
            s.close()


# ---------------------------------------------------------------- 4. scene depth
def scene_depth_cpu(oracle, T, pos, ok):
    """frame_utils::getSceneDepth restated: z of every matched point with the oracle's SE3 transform, nth_element's n/2"""
    z = np.array([oracle.se3_transform(T, p)[2] for p in pos[ok == 1]])
    if len(z) == 0:
        return None
    return np.float32(np.sort(z)[len(z) // 2]), np.float32(0.5 * z.min()), len(z)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
def test_scene_depth_matches_cpu(ctx, oracle, seqs, mode):
    """svob200_tracker_scene_depth against a CPU restatement over points(), the step's T_cur_w and match_ok, bit for bit, after
    every step; sequence 1 has no map point, so its outputs keep what the caller had there."""
    from android_svo_b200 import capi
    cfg = seqs[0][0]
    N = cfg["n_features"]
    n_pt = [N, 0, N]
    src = [seqs[0], seqs[1], seqs[1]]
    take = lambda key, n: np.concatenate([s[3][key][:m] for s, m in zip(src, n)])
    trk = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), 3, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    try:
        trk.set_keyframe(np.stack([s[2][0] for s in src]), np.stack([s[1][0] for s in src]), np.cumsum([0] + n_pt), take("kf_px", n_pt),
                         take("kf_level", n_pt), take("pt_world", n_pt), np.arange(4) * S0, take("seed_px", [S0] * 3), take("seed_level", [S0] * 3))
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([s[2][0] for s in src]))
        off = np.cumsum([0] + n_pt)
        for k in range(1, 5):
            lp = np.concatenate([s[4][k - 1][:m] for s, m in zip(src, n_pt)])
            stats, _, ok = gpu_step(trk, mode, np.stack([s[2][k] for s in src]), np.stack([s[1][k - 1] for s in src]), lp, want_px=True)
            pos = trk.points()[0]
            sentinel_m, sentinel_n = np.float32(-7.25), np.float32(-3.5)
            if mode == "host":
                dm, dn, n = trk.scene_depth(np.full(3, sentinel_m, np.float32), np.full(3, sentinel_n, np.float32))
            else:
                ptrs = [dev_array(ctx, np.full(3, sentinel_m, np.float32)), dev_array(ctx, np.full(3, sentinel_n, np.float32)), dev_array(ctx, np.full(3, -1, np.int32))]
                trk.scene_depth_raw(*ptrs)
                ctx.sync()
                dm, dn, n = np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(3, np.int32)
                for a, p in zip((dm, dn, n), ptrs):
                    ctx.dev_download(a, p)
                    ctx.dev_free(p)
            for b in range(3):
                ref = scene_depth_cpu(oracle, np.array(stats[b]["T_cur_w"]), pos[off[b]:off[b + 1]], ok[off[b]:off[b + 1]])
                if ref is None:
                    assert n[b] == 0 and dm[b] == sentinel_m and dn[b] == sentinel_n, "a sequence without matches was written"
                else:
                    assert n[b] == ref[2] > 80
                    assert dm[b].view(np.uint32) == ref[0].view(np.uint32) and dn[b].view(np.uint32) == ref[1].view(np.uint32), (k, b, dm[b], ref)
    finally:
        trk.close()


# ---------------------------------------------------------------- 5. a keyframe loop without a host round trip
@pytest.mark.gpu
def test_device_keyframe_loop_needs_no_host(ctx, oracle, seqs):
    """Device memory, B = 70 (asynchronous depth filter): step -> scene_depth into device buffers -> a keyframe mask computed
    with torch on the context's stream from device data (the matched-point count of each sequence) -> add_keyframes -> the next
    step, with nothing read back until the end.  The final state equals the same schedule run in host memory."""
    torch = pytest.importorskip("torch")
    from android_svo_b200 import capi
    cfg = seqs[0][0]
    batch, N = 70, cfg["n_features"]
    data = np.arange(batch) % 2
    n_frames = 10

    def rule(n_matched, k):
        return ((n_matched + np.arange(batch) + k) % 4 == 0) if isinstance(n_matched, np.ndarray) else \
            ((n_matched + torch.arange(batch, device=n_matched.device) + k) % 4 == 0)

    def make():
        return make_tracker(ctx, seqs, batch, None, data)

    imgs = np.stack([np.stack([seqs[w][2][k] for w in data]) for k in range(n_frames + 1)])
    T_last = np.stack([np.stack([seqs[w][1][k] for w in data]) for k in range(n_frames + 1)])
    lps = np.stack([np.concatenate([seqs[w][4][k] for w in data]) for k in range(n_frames + 1)])

    # host memory
    h = make()
    n_kfs_host = 0
    try:
        h.set_last(imgs[0])
        dm, dn = np.full(batch, 2.0, np.float32), np.full(batch, 1.0, np.float32)
        for k in range(1, n_frames + 1):
            _, _, ok = h.step(imgs[k], T_last[k - 1], lps[k - 1], want_px=True)
            dm, dn, _ = h.scene_depth(dm, dn)
            m = rule(ok.reshape(batch, N).sum(1), k).astype(np.uint8)
            n_kfs_host += int(m.sum())
            h.add_keyframes(m, dm, dn)
        want = tracker_state(h)
    finally:
        h.close()
    assert 0 < n_kfs_host < batch * n_frames

    d = make()
    try:
        d.set_last_device(imgs[0])
        L = d.L
        stream = torch.cuda.ExternalStream(L.svob200_ctx_stream(ctx.h))
        with torch.cuda.stream(stream):
            g_imgs = torch.from_numpy(imgs).cuda()
            g_T = torch.from_numpy(T_last).cuda()
            g_lp = torch.from_numpy(lps).cuda()
            g_stats = torch.zeros(batch * capi.step_stats_dt.itemsize, dtype=torch.uint8, device="cuda")
            g_px = torch.zeros(batch * N * 2, dtype=torch.float64, device="cuda")
            g_ok = torch.zeros(batch * N, dtype=torch.int32, device="cuda")
            g_dm = torch.full((batch,), 2.0, dtype=torch.float32, device="cuda")
            g_dn = torch.full((batch,), 1.0, dtype=torch.float32, device="cuda")
            g_n = torch.zeros(batch, dtype=torch.int32, device="cuda")
            g_masks = []
            for k in range(1, n_frames + 1):
                rc = L.svob200_tracker_step(d.h, C.c_void_p(g_imgs[k].data_ptr()), cfg["w"], C.c_void_p(g_T[k - 1].data_ptr()),
                                            C.c_void_p(g_lp[k - 1].data_ptr()), C.c_void_p(g_stats.data_ptr()), C.c_void_p(g_px.data_ptr()),
                                            C.c_void_p(g_ok.data_ptr()), capi.MEM_DEVICE)
                ctx._ck(rc)
                d.scene_depth_raw(g_dm.data_ptr(), g_dn.data_ptr(), g_n.data_ptr())
                g_mask = rule(g_ok.view(batch, N).sum(1), k).to(torch.uint8)
                g_masks.append(g_mask)
                d.add_keyframes_raw(g_mask.data_ptr(), g_dm.data_ptr(), g_dn.data_ptr())
        ctx.sync()
        assert sum(int(m.sum()) for m in g_masks) == n_kfs_host
        got = tracker_state(d)
    finally:
        d.close()
    assert got == want


# ---------------------------------------------------------------- 6. argument checks
@pytest.mark.gpu
def test_add_keyframes_and_scene_depth_reject_bad_calls(ctx, seqs):
    """Before set_keyframe or before the first step: SVOB200_ERR_ARG; a bad mem: SVOB200_ERR_ARG; add_keyframes in chain mode:
    SVOB200_ERR_UNSUPPORTED.  Nothing is launched by a rejected call."""
    from android_svo_b200 import capi
    cfg = seqs[0][0]
    f = np.ones(2, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    t = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), 2, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    L = t.L
    try:
        assert L.svob200_tracker_add_keyframes(t.h, None, p(f), p(f), None, None, capi.MEM_HOST) == -1
        assert L.svob200_tracker_scene_depth(t.h, p(f), p(f), None, capi.MEM_HOST) == -1
    finally:
        t.close()
    t = make_tracker(ctx, seqs, 2, None, np.arange(2))
    try:
        t.set_last(np.stack([seqs[w][2][0] for w in range(2)]))
        assert L.svob200_tracker_add_keyframes(t.h, None, p(f), p(f), None, None, capi.MEM_HOST) == -1       # no step yet
        assert L.svob200_tracker_scene_depth(t.h, p(f), p(f), None, capi.MEM_HOST) == -1
        t.step(np.stack([seqs[w][2][1] for w in range(2)]), np.stack([seqs[w][1][0] for w in range(2)]), np.concatenate([seqs[w][4][0] for w in range(2)]))
        n0 = ctx.launch_count()
        for mem in (2, -1):
            assert L.svob200_tracker_add_keyframes(t.h, None, p(f), p(f), None, None, mem) == -1
            assert L.svob200_tracker_scene_depth(t.h, p(f), p(f), None, mem) == -1
        assert L.svob200_tracker_add_keyframes(t.h, None, None, p(f), None, None, capi.MEM_HOST) == -1
        assert ctx.launch_count() == n0
        t.set_chain(30, 120, 1)
        assert L.svob200_tracker_add_keyframes(t.h, None, p(f), p(f), None, None, capi.MEM_HOST) == -4
        assert L.svob200_tracker_add_keyframes(t.h, p(np.ones(2, np.uint8)), p(f), p(f), None, None, capi.MEM_DEVICE) == -4
    finally:
        t.close()


# ---------------------------------------------------------------- 7. the batch-counter limit is per sequence
@pytest.mark.gpu
def test_batch_counter_limit_counts_keyframes_not_calls(ctx, seqs):
    """Calls whose mask selects nobody use up nothing: after 66,000 of them a sequence still takes keyframe batch id 1.  A sequence
    that has taken 65,534 keyframes (Seed::batch_id is 16 bits) is refused, with -1 in both counts and its seeds untouched, while
    the other sequence of the same call takes its keyframe."""
    t = make_tracker(ctx, seqs, 2, None, np.arange(2))
    ptrs = []
    try:
        t.set_last(np.stack([seqs[w][2][0] for w in range(2)]))
        t.step(np.stack([seqs[w][2][1] for w in range(2)]), np.stack([seqs[w][1][0] for w in range(2)]), np.concatenate([seqs[w][4][0] for w in range(2)]))
        ptrs = [dev_array(ctx, a) for a in (np.full(2, 2.0, np.float32), np.full(2, 1.0, np.float32), np.zeros(2, np.uint8), np.array([1, 0], np.uint8))]
        dm, dn, nobody, first = ptrs
        for _ in range(66000):
            t.add_keyframes_raw(nobody, dm, dn)
        n_new, n_drop = t.add_keyframes([0, 1], 2.0, 1.0)
        assert n_new[0] == 0 and n_drop[0] == 0 and n_new[1] > 0
        _, _, _, bt, st = t.seed_refs()
        assert not bt[:CAP][st[:CAP] == 0].any() and bt[CAP:][st[CAP:] == 0].max() == 1
        for _ in range(65534):
            t.add_keyframes_raw(first, dm, dn)
        before = [np.asarray(x)[:CAP].copy() for x in t.seed_refs()] + [t.seeds()[:CAP].tobytes()]
        assert before[3][before[4] == 0].max() == 65534
        n_new, n_drop = t.add_keyframes([1, 1], 2.0, 1.0)
        assert n_new[0] == -1 and n_drop[0] == -1 and n_new[1] > 0 and n_drop[1] == 0
        after = [np.asarray(x)[:CAP] for x in t.seed_refs()] + [t.seeds()[:CAP].tobytes()]
        assert all(np.array_equal(x, y) for x, y in zip(before[:5], after[:5])) and before[5] == after[5]
        _, _, _, bt, st = t.seed_refs()
        assert bt[CAP:][st[CAP:] == 0].max() == 2
    finally:
        t.close()
        for p in ptrs:
            ctx.dev_free(p)
