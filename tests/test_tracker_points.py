"""Point pool of the tracker (svob200_tracker_set_point_pool): a converged seed becomes a candidate point, takes an empty point
slot two steps later, is promoted by a keyframe that matched it and deleted when its keyframe leaves the ring unpromoted
(DepthFilter::updateSeeds -> seed_converged_cb_ -> MapPointCandidates).  The oracle's restatement on the CPU, then the device
against it slot for slot, then the step shapes against each other."""
import numpy as np
import pytest

from oracle.pyoracle import Cam
from point_pool_oracle import PoolSeq
from test_pipeline import KF_DET, gpu_step, make_sequence, seed_matrix
import scenes

N_FRAMES = 13
S0 = 200                              # seeds of the first keyframe
POOL = (3, 2, 3)                      # keyframe ring, max_n_kfs, reseed (the reference's list semantics)
DELETED, CANDIDATE, UNKNOWN = 0, 1, 2
CAP_BIG, CAP_SMALL = 1000, 130       # room for every candidate (the ring evicts some) / a pool that fills up
OFF_IMAGE = -100.0                    # last_px of an empty slot: outside the image, so no alignment patch


def depth_args(k):
    return 2.0 + 0.01 * k, 1.0


def last_px_of(cfg, T_last, pos, ty):
    """the caller's pixel of every live slot in the last frame: its position projected with the last pose"""
    px = np.full((len(ty), 2), OFF_IMAGE)
    live = ty != DELETED
    if live.any():
        from android_svo_b200 import frontend
        px[live] = frontend.project_many(cfg, T_last, pos[live])
    return px


def oracle_seq(data, capacity):
    cfg, poses, imgs, kf, _ = data
    s = PoolSeq(scenes.cam_of(cfg, Cam), cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"], 100.0, 2.4, 1.2, POOL[2], capacity)
    s.set_pool(*POOL); s.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
    s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"][:S0], kf["seed_level"][:S0])
    s.set_last(imgs[0])
    return s


@pytest.fixture(scope="module")
def seqs(oracle):
    return [make_sequence(oracle, "C2", 0x00C0FFEE + 60 + i, N_FRAMES + 1) for i in range(2)]


# ---------------------------------------------------------------- the oracle (CPU)
def test_oracle_point_pool_capacity_zero_changes_nothing(oracle, seqs):
    """A pool without empty slots drops every candidate: poses, matches, seeds and points are those of a sequence without a pool."""
    data = seqs[0]
    cfg, poses, imgs = data[0], data[1], data[2]
    a, b = oracle_seq(data, None), oracle_seq(data, 0)
    try:
        assert a.N == b.N == cfg["n_features"]
        for k in range(1, N_FRAMES + 1):
            pos, ty = a.points()[:2]
            lp = last_px_of(cfg, poses[k - 1], pos, ty)
            ra, rb = a.step(imgs[k], poses[k - 1], lp, want_px=True), b.step(imgs[k], poses[k - 1], lp, want_px=True)
            assert np.array_equal(np.array(ra[0].T_cur_w[:]).view(np.uint64), np.array(rb[0].T_cur_w[:]).view(np.uint64))
            assert np.array_equal(ra[1].view(np.uint64), rb[1].view(np.uint64)) and np.array_equal(ra[2], rb[2])
            if k % 3 == 0:
                assert a.add_keyframe(*depth_args(k)) == b.add_keyframe(*depth_args(k))
            assert np.array_equal(a.seeds().view(np.uint32), b.seeds().view(np.uint32))
            for x, y in zip(a.seed_refs(), b.seed_refs()):
                assert np.array_equal(x, y)
            pa, pb = a.points(), b.points()
            for x, y in zip(pa[:3], pb[:3]):
                assert np.array_equal(x, y)
            assert pa[3] == pa[4] == 0 and pb[4] <= pb[3]
        assert pb[3] > 100 and pb[4] > 0                           # candidates were created, and all that came due dropped
    finally:
        a.close(); b.close()


def se3_inverse(T):
    """float64, written out independently of the oracle: (R^T, -R^T t) of the pose {t, q}"""
    x, y, z, w = T[3:7]
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    return R.T, -R.T @ np.asarray(T[:3])


@pytest.mark.parametrize("capacity", [CAP_BIG, CAP_SMALL])
def test_oracle_candidates_positions_and_order(oracle, seqs, capacity):
    """Every candidate the oracle inserts sits at T_kf_w^-1 * (f / mu) of a seed that converged two steps before, recomputed here
    in float64; the candidates of a step take the empty slots in slot order, in (batch id, seed slot) order; the rest is dropped."""
    data = seqs[0]
    cfg, poses, imgs = data[0], data[1], data[2]
    s = oracle_seq(data, capacity)
    try:
        T_ring = {0: np.asarray(poses[0], np.float64)}              # keyframe index -> pose
        batch_of = {0: 0}                                           # keyframe index -> batch id
        expected = {}                                               # step -> [(batch, slot, kf, pos)] of its converged seeds
        pos, ty, n_obs, created, dropped = s.points()
        n_inserted = n_dropped_full = n_promoted = n_evicted = 0
        for k in range(1, N_FRAMES + 1):
            px_s, lv_s, kf_s, bt_s, st_s = s.seed_refs()
            free_before = np.nonzero(ty == DELETED)[0]
            st, _, ok = s.step(imgs[k], poses[k - 1], last_px_of(cfg, poses[k - 1], pos, ty), want_px=True)
            conv = np.nonzero((s.seed_obs()["status"] == 5) & (st_s == 0))[0]
            mu = s.seeds()[:, 2].astype(np.float64)
            rows = []
            for i in conv:
                f = np.array([(px_s[i, 0] - cfg["cx"]) / cfg["fx"], (px_s[i, 1] - cfg["cy"]) / cfg["fy"], 1.0])
                R, t = se3_inverse(T_ring[kf_s[i]])
                rows.append((bt_s[i], i, kf_s[i], R @ (f / np.linalg.norm(f) / mu[i]) + t))
            expected[k] = sorted(rows, key=lambda r: (r[0], r[1]))
            assert len(rows) == st.n_seeds_converged
            pos2, ty2, n_obs2, created2, dropped2 = s.points()
            assert created2 - created == len(rows)
            # this step inserted the candidates of step k - 2 whose keyframe is still in the ring
            new = np.nonzero((ty == DELETED) & (ty2 == CANDIDATE))[0]
            assert np.array_equal(new, free_before[:len(new)])
            due = [r for r in expected.get(k - 2, []) if batch_of.get(r[2]) == r[0]]
            assert len(new) == min(len(due), len(free_before))
            for slot, r in zip(new, due):
                assert np.allclose(pos2[slot], r[3], rtol=1e-12, atol=1e-12), (k, slot)
            assert (n_obs2[new] == 1).all()
            assert dropped2 - dropped == len(expected.get(k - 2, [])) - len(new)
            n_inserted += len(new); n_dropped_full += len(due) - len(new)
            pos, ty, n_obs, created, dropped = pos2, ty2, n_obs2, created2, dropped2
            if k % 3 == 0:
                s.add_keyframe(*depth_args(k))
                _, _, kf_n, bt_n, st_n = s.seed_refs()
                b_new = bt_n[st_n == 0].max()
                ring = int(kf_n[(st_n == 0) & (bt_n == b_new)][0])
                T_ring[ring] = np.array(st.T_cur_w[:]); batch_of[ring] = int(b_new)
                pos2, ty2, n_obs2, _, _ = s.points()
                cand = ty == CANDIDATE
                n_promoted += int((cand & (ty2 == UNKNOWN)).sum())
                assert ((ty2 == UNKNOWN) == (cand & (ok == 1)) | (ty == UNKNOWN)).all()
                n_evicted += int((cand & (ty2 == DELETED)).sum())
                pos, ty, n_obs = pos2, ty2, n_obs2
        print("capacity %d: inserted %d, dropped for a full pool %d, promoted %d, deleted by eviction %d"
              % (capacity, n_inserted, n_dropped_full, n_promoted, n_evicted))
        assert n_inserted > 0 and n_promoted > 0
        assert n_evicted > 0 if capacity == CAP_BIG else n_dropped_full > 0
    finally:
        s.close()


# ---------------------------------------------------------------- the device (GPU)
def make_tracker(ctx, data, batch, capacity, which):
    from android_svo_b200 import capi
    cfg = data[0][0]
    trk = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), batch, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    trk.set_seed_pool(2400, *POOL); trk.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
    if capacity is not None:
        trk.set_point_pool(capacity)
    N = cfg["n_features"]
    take = lambda key, n=None: np.concatenate([data[w][3][key][:n] for w in which])
    trk.set_keyframe(np.stack([data[w][2][0] for w in which]), np.stack([data[w][1][0] for w in which]), np.arange(batch + 1) * N,
                     take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S0, take("seed_px", S0), take("seed_level", S0))
    return trk


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch,capacity", [("host", 2, CAP_BIG), ("device", 2, CAP_BIG), ("host", 70, CAP_BIG), ("device", 70, CAP_BIG),
                                                 ("device", 70, CAP_SMALL)])
def test_tracker_points_match_oracle(ctx, oracle, seqs, mode, batch, capacity):
    """Device point pool against the pinned oracle (set_pose_override), a keyframe every third frame, slot for slot after every
    step and every keyframe: positions bit for bit, types, observation counts, created / dropped, matches and refined pixels,
    seed states and statuses.  Batch 2 replays a CUDA graph, batch 70 runs the asynchronous depth filter in device memory."""
    which = np.arange(batch) % 2
    cfg = seqs[0][0]
    pinned = [oracle_seq(seqs[d], capacity) for d in range(2)]
    trk = make_tracker(ctx, seqs, batch, capacity, which)
    P = capacity
    try:
        assert trk.P == batch * P and all(s.N == P for s in pinned)
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in which]))
        ev = dict(created=0, inserted=0, promoted=0, evicted=0, dropped=0)

        def compare(k, what):
            pos, ty, no, cr, dr = trk.points()
            seeds_g, obs_g = seed_matrix(trk.seeds()), trk.seed_obs()
            _, _, _, _, st = trk.seed_refs()
            for b in range(batch):
                d = which[b]
                opos, oty, ono, ocr, odr = pinned[d].points()
                sl = slice(b * P, (b + 1) * P)
                assert np.array_equal(bits(pos[sl]), bits(opos)), "positions differ (seq %d, %s %d)" % (b, what, k)
                assert np.array_equal(ty[sl], oty) and np.array_equal(no[sl], ono), "types / observations differ (seq %d, %s %d)" % (b, what, k)
                assert (cr[b], dr[b]) == (ocr, odr), "created / dropped differ (seq %d, %s %d)" % (b, what, k)
                So = pinned[d].num_slots()
                ssl = slice(b * 2400, b * 2400 + So)
                ost = pinned[d].seed_refs()[4]
                assert np.array_equal(st[ssl], ost)
                alive = ost == 0
                assert np.array_equal(seeds_g[ssl][alive].view(np.uint32), pinned[d].seeds()[alive].view(np.uint32)), "seeds differ (seq %d, %s %d)" % (b, what, k)
                assert np.array_equal(obs_g["status"][ssl], pinned[d].seed_obs()["status"])
            return pinned[0].points()

        o_ty = pinned[0].points()[1]
        for k in range(1, N_FRAMES + 1):
            lp = [last_px_of(cfg, seqs[d][1][k - 1], *pinned[d].points()[:2]) for d in range(2)]
            stats, px_g, ok_g = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                                         np.concatenate([lp[w] for w in which]), want_px=True)
            for d in range(2):
                pinned[d].set_pose_override(stats[d]["T_cur_w"])
                _, px_o, ok_o = pinned[d].step(seqs[d][2][k], seqs[d][1][k - 1], lp[d], want_px=True)
                for b in np.nonzero(which == d)[0]:
                    assert np.array_equal(ok_g[b * P:(b + 1) * P], ok_o) and np.array_equal(bits(px_g[b * P:(b + 1) * P]), bits(px_o)), \
                        "matches differ (seq %d, frame %d)" % (b, k)
            pos, ty, no, cr, dr = compare(k, "frame")
            ev["inserted"] += int(((o_ty == DELETED) & (ty == CANDIDATE)).sum())
            o_ty = ty
            if k % 3 == 0:
                n_new, _ = trk.add_keyframe(*depth_args(k))
                for d in range(2):
                    assert (n_new[which == d] == pinned[d].add_keyframe(*depth_args(k))).all()
                pos, ty, no, cr, dr = compare(k, "keyframe")
                ev["promoted"] += int(((o_ty == CANDIDATE) & (ty == UNKNOWN)).sum())
                ev["evicted"] += int(((o_ty == CANDIDATE) & (ty == DELETED)).sum())
                o_ty = ty
        ev["created"], ev["dropped"] = cr, dr
        print("point pool, sequence 0:", ev)
        assert ev["created"] > 100 and ev["inserted"] > 0 and ev["promoted"] > 0
        assert ev["evicted"] > 0 if capacity == CAP_BIG else ev["dropped"] > 0
    finally:
        trk.close()
        for s in pinned:
            s.close()


@pytest.mark.gpu
def test_tracker_points_shapes_identical(ctx, oracle, seqs):
    """The same inputs through every step shape give byte-identical step records, matches and point tables: host memory at
    B = 300 (two chunks), device memory at B = 70 (asynchronous depth filter) and B = 70 with profiling (in place); device
    memory at B = 3 (graph replay) and host memory at B = 3 with profiling (in place).  The two groups differ in how sparse
    alignment spreads a problem (one CTA per sequence above 16 sequences, a cluster of CTAs below): its double sums are
    tolerance-matched across that choice (DESIGN section 3), so each group is compared within itself."""
    cfg = seqs[0][0]
    groups = [[("host", 300, False), ("device", 70, False), ("device", 70, True)], [("device", 3, False), ("host", 3, True)]]
    inputs = {}

    def run(mode, batch, prof):
        which = np.arange(batch) % 2
        trk = make_tracker(ctx, seqs, batch, CAP_BIG, which)
        out = []
        try:
            if prof:
                trk.enable_profiling(True)
            (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in which]))
            for k in range(1, N_FRAMES + 1):
                if k not in inputs:                       # the caller's pixels, from the first run's point table
                    pos, ty = trk.points()[:2]
                    inputs[k] = [last_px_of(cfg, seqs[d][1][k - 1], pos[d * CAP_BIG:(d + 1) * CAP_BIG], ty[d * CAP_BIG:(d + 1) * CAP_BIG])
                                 for d in range(2)]
                stats, px, ok = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                                         np.concatenate([inputs[k][w] for w in which]), want_px=True)
                if k % 3 == 0:
                    trk.add_keyframe(*depth_args(k))
                pos, ty, no, cr, dr = trk.points()
                out.append(dict(stats=stats, px=px, ok=ok, pos=pos, ty=ty, no=no, cr=cr, dr=dr))
        finally:
            trk.close()
        return out

    for group in groups:
        ref = run(*group[0])
        assert ref[-1]["cr"].min() > 100 and (ref[-1]["ty"] == UNKNOWN).sum() > group[0][1] * cfg["n_features"]
        for mode, batch, prof in group[1:]:
            P = batch * CAP_BIG
            for k, (a, b) in enumerate(zip(run(mode, batch, prof), ref), 1):
                tag = "%s B=%d profiling=%s against %s B=%d, frame %d" % (mode, batch, prof, group[0][0], group[0][1], k)
                assert a["stats"].tobytes() == b["stats"][:batch].tobytes(), tag
                assert bits(a["px"]).tobytes() == bits(b["px"][:P]).tobytes() and a["ok"].tobytes() == b["ok"][:P].tobytes(), tag
                assert bits(a["pos"]).tobytes() == bits(b["pos"][:P]).tobytes(), tag
                assert np.array_equal(a["ty"], b["ty"][:P]) and np.array_equal(a["no"], b["no"][:P]), tag
                assert np.array_equal(a["cr"], b["cr"][:batch]) and np.array_equal(a["dr"], b["dr"][:batch]), tag


@pytest.mark.gpu
def test_tracker_point_pool_validation(ctx, seqs):
    """set_point_pool after set_keyframe or with a negative capacity is rejected; chain mode refuses a pool; without a pool the
    slot count is the set_keyframe point count and no candidate is counted.  With unequal counts per sequence, the point and
    seed slots right after set_keyframe equal the caller's arrays laid out in numpy."""
    from android_svo_b200 import capi
    cfg = seqs[0][0]
    which = np.arange(2)
    t0 = make_tracker(ctx, seqs, 2, None, which)
    try:
        assert t0.P == 2 * cfg["n_features"]
        pos, ty, no, cr, dr = t0.points()
        assert (ty == UNKNOWN).all() and (no == 1).all() and not cr.any() and not dr.any()
        with pytest.raises(capi.Svob200Error):
            t0.set_point_pool(10)
    finally:
        t0.close()
    t1 = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), 2, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    try:
        with pytest.raises(capi.Svob200Error):
            t1.set_point_pool(-1)
    finally:
        t1.close()
    t2 = make_tracker(ctx, seqs, 2, 150, which)
    try:
        assert t2.P == 2 * 150
        pos, ty, no, cr, dr = t2.points()
        assert (ty[:cfg["n_features"]] == UNKNOWN).all() and (ty[cfg["n_features"]:150] == DELETED).all() and (no[cfg["n_features"]:150] == 0).all()
        rc = t2.L.svob200_tracker_set_chain(t2.h, 30, 120, 1)
        assert rc == -4                                            # SVOB200_ERR_UNSUPPORTED
    finally:
        t2.close()
    # unequal counts per sequence (one without map points, one without seeds), pool capacities above and below them: right after
    # set_keyframe each sequence's slots hold its map points / seeds in order, then empty slots
    n_pt, n_sd, cap_pt, cap_sd = [cfg["n_features"], 0, 37, 90], [S0, 50, 0, 7], 100, 60
    src = [seqs[b % 2] for b in range(4)]
    take = lambda key, n: np.concatenate([src[b][3][key][:n[b]] for b in range(4)])
    t3 = capi.Tracker(ctx, scenes.cam_of(cfg, capi.Camera), 4, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    try:
        t3.set_seed_pool(cap_sd, *POOL)
        t3.set_point_pool(cap_pt)
        t3.set_keyframe(np.stack([s[2][0] for s in src]), np.stack([s[1][0] for s in src]), np.cumsum([0] + n_pt), take("kf_px", n_pt),
                        take("kf_level", n_pt), take("pt_world", n_pt), np.cumsum([0] + n_sd), take("seed_px", n_sd), take("seed_level", n_sd))

        def slots(key, n, cap, width):
            return np.concatenate([np.concatenate([np.asarray(src[b][3][key], np.float64)[:n[b]].reshape(-1, width), np.zeros((max(n[b], cap) - n[b], width))])
                                   for b in range(4)])
        real_pt = np.concatenate([np.arange(max(n, cap_pt)) < n for n in n_pt])
        real_sd = np.concatenate([np.arange(max(n, cap_sd)) < n for n in n_sd])
        assert t3.P == len(real_pt) == 120 + 3 * 100 and t3.S == len(real_sd) == S0 + 3 * 60
        pos, ty, no, cr, dr = t3.points()
        assert np.array_equal(bits(pos), bits(slots("pt_world", n_pt, cap_pt, 3)))
        assert np.array_equal(ty, np.where(real_pt, UNKNOWN, DELETED)) and np.array_equal(no, real_pt) and not cr.any() and not dr.any()
        px, lv, kf, bt, st = t3.seed_refs()
        assert np.array_equal(bits(px), bits(slots("seed_px", n_sd, cap_sd, 2))) and np.array_equal(lv, slots("seed_level", n_sd, cap_sd, 1)[:, 0])
        assert not kf.any() and not bt.any() and np.array_equal(st, ~real_sd)
    finally:
        t3.close()
