"""Per-frame front-end step (pyramid -> sparse align -> reprojection refinement -> seed update):
the C restatement against the real reference (CPU), and svob200_tracker_step against the C
restatement (GPU)."""
import numpy as np
import pytest

from android_svo_b200 import synth, frontend
from oracle.pyoracle import Cam, OracleSeq, RefSeq
import scenes


def recycle(cells, thr, n):
    """cells above thr, recycled when the view holds fewer than n (full-size configs: same load as the bench)"""
    good = cells[cells["score"].astype(np.float64) > thr]
    out = np.resize(good, n) if len(good) < n else good[:n]
    # keyframe_setup takes the first n cells above thr: hand it exactly those, with scores that pass
    out = out.copy(); out["score"] = np.maximum(out["score"], np.float32(thr + 1))
    return out


def make_sequence(oracle, name, seed, n_frames, tex_size=1024, stride=3, allow_recycle=False):
    cfg = synth.CONFIGS[name]
    poses = synth.trajectory(n_frames * stride, seed=seed)[::stride]
    tex = scenes.texture(tex_size)
    imgs = [synth.render(tex, cfg, T) for T in poses]
    fc, ft, sc, st = frontend.DETECT[name]
    pyr = oracle.pyramid(imgs[0], cfg["n_levels"])
    _, fcells = oracle.fast_detect(pyr, cfg["n_pyr"], fc, ft)
    _, scells = oracle.fast_detect(pyr, cfg["n_pyr"], sc, st)
    if allow_recycle:
        fcells, scells = recycle(fcells, ft, cfg["n_features"]), recycle(scells, st, cfg["n_seeds"])
    kf = frontend.keyframe_setup(cfg, poses[0], fcells, scells, ft, st)
    last_px = [frontend.project_many(cfg, poses[k], kf["pt_world"]) for k in range(n_frames)]
    return cfg, poses, imgs, kf, last_px


def test_oracle_step_matches_reference(oracle, ref):
    """The C restatement against the reference's own classes over a sequence: BIT-identical poses, refined pixels and
    seed states (the restatement keeps the reference's summation order and Eigen's LDLT association)."""
    cfg, poses, imgs, kf, last_px = make_sequence(oracle, "C2", 0x00C0FFEE, 11)
    cam = scenes.cam_of(cfg, Cam)
    args = (cam, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    so, sr = OracleSeq(oracle, *args), RefSeq(ref, *args)
    try:
        for s in (so, sr):
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"])
            s.set_last(imgs[0])
        total_conv = 0
        for k in range(1, 11):
            a, pxa, oka = so.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            b, pxb, okb = sr.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            assert a.n_tracked == b.n_tracked and a.align_iters == b.align_iters
            assert np.array_equal(np.array(a.T_cur_w[:]), np.array(b.T_cur_w[:])), "pose not bit-identical at frame %d" % k
            assert a.n_matched == b.n_matched and np.array_equal(oka, okb)
            assert np.array_equal(pxa, pxb)
            assert a.n_seeds_converged == b.n_seeds_converged        # (the reference harness reports the callback count only)
            assert np.array_equal(so.seeds().view(np.uint32), sr.seeds().view(np.uint32)), "seed states not bit-identical after frame %d" % k
            total_conv += a.n_seeds_converged
            # sanity: alignment recovers the true pose to a few mm (stops at level 2)
            grot, gtrans = synth.pose_error(np.array(a.T_cur_w[:]), poses[k])
            assert grot < 1e-2 and gtrans < 3e-2
            assert a.n_tracked > 90 and a.n_matched > 90
        assert total_conv > 150
    finally:
        so.close(); sr.close()


SEED_COLS = ("a", "b", "mu", "z_range", "sigma2")
OBS_DISCRETE = ("status", "search_level", "zmssd_best", "n_evals")


def seed_matrix(rec):
    return np.stack([rec[c] for c in SEED_COLS], 1)


def gpu_step(trk, mode, *a, **kw):
    """mode 'host': SVOB200_MEM_HOST (staged copies, chunked);  'device': SVOB200_MEM_DEVICE — level 0 aliases the
    caller's device buffer, the whole batch is one range (a forked CUDA graph for batches <= 64): what bench.py's `value` times"""
    return (trk.step if mode == "host" else trk.step_device)(*a, **kw)


class SeedParity:
    """Seed-state comparison with the cause of every deviation named (DESIGN.md section 4).

    The device sums sparse alignment's H / Jres in a different order than the reference, so its pose differs by ~1e-10
    (tolerance-matched, SURVEY 8a a7).  Everything after the pose is restated operation by operation, so with the SAME pose
    the depth filter must reproduce the oracle's bits (only a double libm ulp that survives the cast to float could differ).
    Hence two oracles per sequence:
      free     runs on its own aligned pose -> value tolerance 1e-5 relative; seeds outside it are COUNTED, and each one must be
               reproduced bit for bit by the pinned oracle (i.e. the deviation is the 1e-10 pose difference moving a float
               rounding of 1/z or tau^2, amplified by the cancellation in sigma2 = C1(s2+m^2) + C2(sigma2+mu^2) - mu_new^2)
      pinned   gets the device's pose injected -> discrete decisions and seed bits must be IDENTICAL (count asserted 0)
    Under the pinned pose the observations themselves are compared too: epi_length bit-exact wherever the matcher ran, the
    triangulated depth z within 1e-12 relative wherever a seed was updated.  In the young-seed regime (every seed reset to its
    prior after each frame) equal seed states prove little; the observations carry the information."""

    def __init__(self):
        self.n_seeds = self.n_outside_tol = self.n_pinned_bit_diff = self.n_discrete_diff = self.n_free_discrete_diff = 0
        self.n_evals = self.n_long_walks = 0

    def check(self, seeds_gpu, obs_gpu, free, pinned):
        sg = seed_matrix(seeds_gpu)
        sf, sp = free.seeds(), pinned.seeds()
        of, op = free.seed_obs(), pinned.seed_obs()
        self.n_seeds += len(sg)
        # pinned pose: identical decisions, identical observation, identical bits
        for key in OBS_DISCRETE:
            self.n_discrete_diff += int((obs_gpu[key] != op[key]).sum())
            self.n_free_discrete_diff += int((obs_gpu[key] != of[key]).sum())
        upd = obs_gpu["status"] >= 3
        assert np.array_equal(obs_gpu["px_cur"][upd], op["px_cur"][upd]), "matched pixel differs under the same pose"
        assert np.array_equal(obs_gpu["epi_length"][upd].view(np.uint64), op["epi_length"][upd].view(np.uint64)), \
            "epipolar segment length differs under the same pose"
        tri = (obs_gpu["status"] >= 4) & (op["status"] >= 4)
        assert np.all(np.abs(obs_gpu["z"][tri] - op["z"][tri]) <= 1e-12 * np.abs(op["z"][tri])), "triangulated depth differs under the same pose"
        self.n_evals += int(obs_gpu["n_evals"].sum())
        self.n_long_walks += int((upd & (obs_gpu["epi_length"] / 0.7 > 64)).sum())
        bit_diff = (sg.view(np.uint32) != sp.view(np.uint32)).any(axis=1)
        self.n_pinned_bit_diff += int(bit_diff.sum())
        # own pose: 1e-5 relative, deviations counted and each explained by the pinned oracle
        outside = ~np.isclose(sg, sf, rtol=1e-5, atol=0).all(axis=1)
        self.n_outside_tol += int(outside.sum())
        assert not (outside & bit_diff).any(), "a seed deviates from the oracle beyond 1e-5 and the pose difference does not explain it"
        assert np.allclose(sg, sf, rtol=2e-2, atol=0), "a seed deviates grossly from the free-running oracle"

    def mean_evals(self):
        return self.n_evals / max(self.n_seeds, 1)

    def finish(self, max_outside_frac=0.01):
        print("seed parity: %d seed-frames, %d outside 1e-5 vs the free-running oracle (all reproduced bit-exactly under the device's pose), "
              "%d bit differences / %d discrete differences under the same pose, %d discrete differences vs the free-running oracle; "
              "mean n_evals %.2f, %d walks longer than 64 samples"
              % (self.n_seeds, self.n_outside_tol, self.n_pinned_bit_diff, self.n_discrete_diff, self.n_free_discrete_diff,
                 self.mean_evals(), self.n_long_walks))
        assert self.n_discrete_diff == 0, "%d discrete seed decisions differ under the same pose" % self.n_discrete_diff
        assert self.n_pinned_bit_diff == 0, "%d seeds differ in bits under the same pose" % self.n_pinned_bit_diff
        assert self.n_outside_tol <= max_outside_frac * self.n_seeds

    def assert_young(self):
        """the regime really is young: far more ZMSSD evaluations per seed than the steady regime's 2.6, and long walks"""
        assert self.mean_evals() > 2 * 2.6 and self.n_long_walks > 0, (self.mean_evals(), self.n_long_walks)


# bench.py --seed-regime: steady re-initialises finished seeds (the defaults), young re-initialises every seed after every frame
# to a wide prior (reseed = 2, depth_min = 0.3)
REGIMES = {"steady": (100.0, 2.4, 1.2, 1), "young": (100.0, 2.4, 0.3, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("regime", ["steady", "young"])
@pytest.mark.parametrize("name,batch,n_frames", [("C2", 3, 10), ("C3", 2, 4), ("C2", 1, 6), ("C2", 70, 4)])
def test_tracker_step_matches_oracle(ctx, oracle, name, batch, n_frames, mode, regime):
    """svob200_tracker_step against the oracle, in both seed regimes of bench.py.  A batch above 64 runs direct launches, the
    asynchronous depth filter and a two-wave search grid; it replicates 3 distinct sequences, and every replica must return
    the bit-identical step record, refined pixels, seed state and seed observations of its first copy."""
    from android_svo_b200 import capi
    n_distinct = min(batch, 3)
    seqs = [make_sequence(oracle, name, 0x00C0FFEE + i, n_frames + 1) for i in range(n_distinct)]
    which = np.arange(batch) % n_distinct
    cfg = seqs[0][0]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    free = [OracleSeq(oracle, cam_o, *args, *REGIMES[regime]) for _ in range(n_distinct)]
    pinned = [OracleSeq(oracle, cam_o, *args, *REGIMES[regime]) for _ in range(n_distinct)]
    trk = capi.Tracker(ctx, cam_g, batch, *args, *REGIMES[regime])
    par = SeedParity()
    try:
        N, S = cfg["n_features"], cfg["n_seeds"]
        for grp in (free, pinned):
            for s, (_, poses, imgs, kf, _) in zip(grp, seqs):
                s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"])
                s.set_last(imgs[0])
        cat = lambda key: np.concatenate([seqs[w][3][key] for w in which])
        trk.set_keyframe(np.stack([seqs[w][2][0] for w in which]), np.stack([seqs[w][1][0] for w in which]), np.arange(batch + 1) * N,
                         cat("kf_px"), cat("kf_level"), cat("pt_world"), np.arange(batch + 1) * S, cat("seed_px"), cat("seed_level"))
        if mode == "host":
            trk.set_last(np.stack([seqs[w][2][0] for w in which]))
        else:
            trk.set_last_device(np.stack([seqs[w][2][0] for w in which]))
        for k in range(1, n_frames + 1):
            stats, px, ok = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                                     np.concatenate([seqs[w][4][k - 1] for w in which]), want_px=True)
            seeds_g, obs_g = trk.seeds(), trk.seed_obs()
            for b in range(n_distinct, batch):
                d = which[b]
                assert stats[b].tobytes() == stats[d].tobytes(), "replica %d of sequence %d: step record differs" % (b, d)
                assert np.array_equal(px[b * N:(b + 1) * N], px[d * N:(d + 1) * N]) and np.array_equal(ok[b * N:(b + 1) * N], ok[d * N:(d + 1) * N])
                assert seeds_g[b * S:(b + 1) * S].tobytes() == seeds_g[d * S:(d + 1) * S].tobytes()
                assert obs_g[b * S:(b + 1) * S].tobytes() == obs_g[d * S:(d + 1) * S].tobytes()
            for b in range(n_distinct):
                g = stats[b]
                e, pxe, oke = free[b].step(seqs[b][2][k], seqs[b][1][k - 1], seqs[b][4][k - 1], want_px=True)
                pinned[b].set_pose_override(g["T_cur_w"])
                p, pxp, okp = pinned[b].step(seqs[b][2][k], seqs[b][1][k - 1], seqs[b][4][k - 1], want_px=True)
                assert g["n_tracked"] == e.n_tracked
                assert g["align_iters"] == e.align_iters, "GN iteration count differs (decision flip)"
                rot, trans = synth.pose_error(g["T_cur_w"], np.array(e.T_cur_w[:]))
                assert rot <= 1e-4 and trans <= 2e-4
                assert rot < 1e-9 and trans < 1e-9
                sl = slice(b * N, (b + 1) * N)
                assert g["n_matched"] == e.n_matched and np.array_equal(ok[sl], oke)
                assert np.abs(px[sl] - pxe).max() <= 1e-3
                # same pose -> the refined pixels are bit-identical
                assert np.array_equal(ok[sl], okp) and np.array_equal(px[sl], pxp)
                for key in ("n_seeds_updated", "n_seeds_converged", "n_seeds_failed", "n_seeds_skipped"):
                    assert g[key] == getattr(p, key), key
                par.check(seeds_g[b * S:(b + 1) * S], obs_g[b * S:(b + 1) * S], free[b], pinned[b])
        par.finish()
        if regime == "young":
            par.assert_young()
    finally:
        trk.close()
        for s in free + pinned:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [0, 1])
@pytest.mark.parametrize("batch", [1, 3, 70, 300])
def test_tracker_device_mode_bit_identical_to_host_mode(ctx, oracle, batch, chain):
    """SVOB200_MEM_DEVICE (frame_bind aliasing, forked CUDA graph for batch <= 64, plain launches above) must return the
    bit-identical step record, refined pixels, seed state and seed observations as SVOB200_MEM_HOST on the same inputs.
    A host-memory batch of 300 runs in two chunks, 256 + 44."""
    from android_svo_b200 import capi
    n_frames, n_distinct = 6, min(batch, 3)
    seqs = [make_sequence(oracle, "C2", 0x00C0FFEE + 40 + i, n_frames + 1) for i in range(n_distinct)]
    which = np.arange(batch) % n_distinct
    cfg = seqs[0][0]
    cam_g = scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    N, S = cfg["n_features"], cfg["n_seeds"]
    out = {}
    for mode in ("host", "device"):
        trk = capi.Tracker(ctx, cam_g, batch, *args)
        try:
            take = lambda key: np.concatenate([seqs[w][3][key] for w in which])
            trk.set_keyframe(np.stack([seqs[w][2][0] for w in which]), np.stack([seqs[w][1][0] for w in which]), np.arange(batch + 1) * N,
                             take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S, take("seed_px"), take("seed_level"))
            if chain:
                trk.set_chain(30, 40, 1)
            (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in which]))
            rec = []
            for k in range(1, n_frames + 1):
                stats, px, ok = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                                         np.concatenate([seqs[w][4][k - 1] for w in which]), want_px=True)
                rec.append((stats.copy(), px.copy(), ok.copy(), trk.seeds().copy(), trk.seed_obs().copy()))
            out[mode] = rec
        finally:
            trk.close()
    for k, (h, d) in enumerate(zip(out["host"], out["device"])):
        for name, x, y in zip(("stats", "px", "ok", "seeds", "seed_obs"), h, d):
            assert x.tobytes() == y.tobytes(), "%s differs between host and device mode at frame %d" % (name, k + 1)
    assert out["host"][-1][0]["n_matched"].min() > 20


@pytest.mark.gpu
def test_tracker_step_full_size_c4(ctx, oracle):
    """BASELINE.json configs[3] at its full size: one 1920x1080 sequence, 5-level pyramid, 1,000 features, 10,000 seeds,
    two frames against the oracle (sparse align runs on a thread-block cluster at this batch size), resident path."""
    from android_svo_b200 import capi
    cfg, poses, imgs, kf, last_px = make_sequence(oracle, "C4", 0x00C0FFEE + 9, 3, tex_size=2048, allow_recycle=True)
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    N, S = cfg["n_features"], cfg["n_seeds"]
    assert (N, S) == (1000, 10000)
    so, sp = OracleSeq(oracle, cam_o, *args), OracleSeq(oracle, cam_o, *args)
    trk = capi.Tracker(ctx, cam_g, 1, *args)
    par = SeedParity()
    try:
        for s in (so, sp):
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"]); s.set_last(imgs[0])
        trk.set_keyframe(imgs[0][None], poses[0][None], [0, N], kf["kf_px"], kf["kf_level"], kf["pt_world"], [0, S], kf["seed_px"], kf["seed_level"])
        trk.set_last_device(imgs[0][None])
        for k in (1, 2):
            stats, px, ok = trk.step_device(imgs[k][None], poses[k - 1][None], last_px[k - 1], want_px=True)
            e, pxe, oke = so.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            g = stats[0]
            sp.set_pose_override(g["T_cur_w"])
            p, pxp, okp = sp.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            assert g["n_tracked"] == e.n_tracked and g["align_iters"] == e.align_iters
            rot, trans = synth.pose_error(g["T_cur_w"], np.array(e.T_cur_w[:]))
            assert rot < 1e-9 and trans < 1e-9
            assert g["n_matched"] == e.n_matched and np.array_equal(ok, oke) and np.abs(px - pxe).max() <= 1e-3
            assert np.array_equal(ok, okp) and np.array_equal(px, pxp)
            for key in ("n_seeds_updated", "n_seeds_converged", "n_seeds_failed", "n_seeds_skipped"):
                assert g[key] == getattr(p, key), key
            par.check(trk.seeds(), trk.seed_obs(), so, sp)
        par.finish()
    finally:
        trk.close(); so.close(); sp.close()


@pytest.mark.gpu
def test_tracker_c5_size_replicas(ctx, oracle):
    """BASELINE.json configs[4] at its full size (4,096 sequences in one batch) through a size-independent property:
    the batch holds 32 distinct sequences, each replicated 128 times at scattered batch positions; every replica must
    return the bit-identical step record, refined pixels, seed state and seed observations (no cross-talk, no dependence
    on the position in the batch or on which SM / group processed it), and replica 0 of each sequence must match the oracle.
    Runs the EXACT path bench.py's `value` times — SVOB200_MEM_DEVICE: level-0 aliasing + ONE 4,096-wide
    range (491 k candidates, 3.1 M seeds per launch) — and the SVOB200_MEM_HOST path (16 chunks of 256 on a copy stream):
    the two must agree bit for bit.  Four steps, so that the frame slot the asynchronous depth filter searches is reused while
    that filter runs; in both seed regimes of bench.py."""
    from android_svo_b200 import capi
    n_distinct, B, n_steps = 32, 4096, 4
    seqs = [make_sequence(oracle, "C2", 0x00C0FFEE + 100 + i, n_steps + 1) for i in range(n_distinct)]
    cfg = seqs[0][0]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    N, S = cfg["n_features"], cfg["n_seeds"]
    which = (np.arange(B) * 13) % n_distinct                      # scattered assignment of sequences to batch slots
    take = lambda key: np.concatenate([seqs[w][3][key] for w in which])
    frames = [np.stack([seqs[w][2][k] for w in which]) for k in range(n_steps + 1)]
    for regime in ("steady", "young"):
        res, device_poses = {}, []
        for mode in ("device", "host"):
            trk = capi.Tracker(ctx, cam_g, B, *args, *REGIMES[regime])
            try:
                trk.set_keyframe(frames[0], np.stack([seqs[w][1][0] for w in which]), np.arange(B + 1) * N,
                                 take("kf_px"), take("kf_level"), take("pt_world"), np.arange(B + 1) * S, take("seed_px"), take("seed_level"))
                (trk.set_last if mode == "host" else trk.set_last_device)(frames[0])
                for k in range(1, n_steps + 1):
                    stats, px, ok = gpu_step(trk, mode, frames[k], np.stack([seqs[w][1][k - 1] for w in which]),
                                             np.concatenate([seqs[w][4][k - 1] for w in which]), want_px=True)
                    if mode == "device":
                        device_poses.append(stats["T_cur_w"].copy())
                res[mode] = (stats, px, ok, trk.seeds(), trk.seed_obs())
            finally:
                trk.close()
        for name, x, y in zip(("stats", "px", "ok", "seeds", "seed_obs"), res["device"], res["host"]):
            assert x.tobytes() == y.tobytes(), "%s: %s differs between the one-range device path and the chunked host path" % (regime, name)
        stats, px, ok, seeds_flat, obs_flat = res["device"]
        px = px.reshape(B, N, 2); ok = ok.reshape(B, N)
        seeds, obs = seed_matrix(seeds_flat).reshape(B, S, 5), obs_flat.reshape(B, S)
        for d in range(n_distinct):
            idx = np.nonzero(which == d)[0]
            first = idx[0]
            for name in stats.dtype.names:
                assert (stats[name][idx] == stats[name][first]).all(), "%s: replicas of sequence %d differ in %s" % (regime, d, name)
            assert (px[idx] == px[first]).all() and (ok[idx] == ok[first]).all()
            assert (seeds[idx].view(np.uint32) == seeds[first].view(np.uint32)).all()
            assert all(obs[i].tobytes() == obs[first].tobytes() for i in idx)
        par = SeedParity()
        for d in range(0, n_distinct, 8):                      # a few against the oracle: free-running, and pinned to the device's poses
            so, sp = OracleSeq(oracle, cam_o, *args, *REGIMES[regime]), OracleSeq(oracle, cam_o, *args, *REGIMES[regime])
            try:
                _, poses, imgs, kf, last_px = seqs[d]
                first = np.nonzero(which == d)[0][0]
                for s in (so, sp):
                    s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"]); s.set_last(imgs[0])
                for k in range(1, n_steps + 1):
                    e, pxe, oke = so.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
                    sp.set_pose_override(device_poses[k - 1][first])
                    p = sp.step(imgs[k], poses[k - 1], last_px[k - 1])
                g = stats[first]
                rot, trans = synth.pose_error(g["T_cur_w"], np.array(e.T_cur_w[:]))
                assert rot < 1e-9 and trans < 1e-9 and g["n_matched"] == e.n_matched and g["n_seeds_updated"] == p.n_seeds_updated, regime
                assert np.array_equal(ok[first], oke) and np.abs(px[first] - pxe).max() <= 1e-3, regime
                par.check(seeds_flat[first * S:(first + 1) * S], obs_flat[first * S:(first + 1) * S], so, sp)
            finally:
                so.close(); sp.close()
        par.finish()
        if regime == "young":
            # (the tracker-step test asserts the long walks; these four sequences need not have one in four steps)
            assert par.mean_evals() > 2 * 2.6, par.mean_evals()


def test_oracle_chain_matches_reference(oracle, ref):
    """Chain mode: Reprojector::reprojectMap + pose_optimizer::optimizeGaussNewton between alignment and the depth filter,
    as FrameHandlerMono::processFrame runs them (frame_handler_mono.cpp:191-222) — the oracle's restatement against the
    reference's own classes over a sequence (per-point reprojection counters reset every frame on both sides)."""
    cfg, poses, imgs, kf, last_px = make_sequence(oracle, "C2", 0x00C0FFEE + 3, 8)
    cam = scenes.cam_of(cfg, Cam)
    args = (cam, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    so, sr = OracleSeq(oracle, *args), RefSeq(ref, *args)
    try:
        for s in (so, sr):
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"])
            s.set_chain(30, 120, 1)
            s.set_last(imgs[0])
        for k in range(1, 8):
            a, pxa, oka = so.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            b, pxb, okb = sr.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            assert a.n_tracked == b.n_tracked and a.align_iters == b.align_iters
            assert (a.n_matched, a.n_reproj_trials, a.n_pose_obs) == (b.n_matched, b.n_reproj_trials, b.n_pose_obs)
            assert np.array_equal(oka, okb) and np.array_equal(pxa[oka == 1], pxb[okb == 1])     # the frame's new features: bit-exact
            assert np.array_equal(np.array(a.T_cur_w[:]), np.array(b.T_cur_w[:]))                # pose after the optimiser: bit-exact
            assert a.n_seeds_converged == b.n_seeds_converged
            assert np.array_equal(so.seeds().view(np.uint32), sr.seeds().view(np.uint32))
            # the pose optimiser tightens the alignment pose (which stops at level 2) against the ground truth
            grot, gtrans = synth.pose_error(np.array(a.T_cur_w[:]), poses[k])
            assert grot < 2e-3 and gtrans < 6e-3 and 40 < a.n_matched <= 121
    finally:
        so.close(); sr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("pose_opt", [1, 0])
def test_tracker_chain_matches_oracle(ctx, oracle, pose_opt, mode):
    """svob200_tracker_step in chain mode (reprojector grid rules + pose optimiser inside the step) against the oracle's
    chain, which is bit-exact to the reference's (test_oracle_chain_matches_reference).  Seeds: SeedParity (the pinned oracle
    gets the device's pose after its optimiser for the depth filter)."""
    from android_svo_b200 import capi
    batch, n_frames = 3, 5
    seqs = [make_sequence(oracle, "C2", 0x00C0FFEE + 20 + i, n_frames + 1) for i in range(batch)]
    cfg = seqs[0][0]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    free = [OracleSeq(oracle, cam_o, *args) for _ in range(batch)]
    pinned = [OracleSeq(oracle, cam_o, *args) for _ in range(batch)]
    trk = capi.Tracker(ctx, cam_g, batch, *args)
    par = SeedParity()
    try:
        N, S = cfg["n_features"], cfg["n_seeds"]
        for grp in (free, pinned):
            for s, (_, poses, imgs, kf, _) in zip(grp, seqs):
                s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"])
                s.set_chain(30, 40, pose_opt)                       # max_fts = 40: the break fires
                s.set_last(imgs[0])
        cat = lambda key: np.concatenate([q[3][key] for q in seqs])
        trk.set_keyframe(np.stack([q[2][0] for q in seqs]), np.stack([q[1][0] for q in seqs]), np.arange(batch + 1) * N,
                         cat("kf_px"), cat("kf_level"), cat("pt_world"), np.arange(batch + 1) * S, cat("seed_px"), cat("seed_level"))
        trk.set_chain(30, 40, pose_opt)
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([q[2][0] for q in seqs]))
        for k in range(1, n_frames + 1):
            stats, px, ok = gpu_step(trk, mode, np.stack([q[2][k] for q in seqs]), np.stack([q[1][k - 1] for q in seqs]),
                                     np.concatenate([q[4][k - 1] for q in seqs]), want_px=True)
            seeds_g, obs_g = trk.seeds(), trk.seed_obs()
            for b in range(batch):
                g = stats[b]
                e, pxe, oke = free[b].step(seqs[b][2][k], seqs[b][1][k - 1], seqs[b][4][k - 1], want_px=True)
                pinned[b].set_pose_override(g["T_cur_w"])
                p = pinned[b].step(seqs[b][2][k], seqs[b][1][k - 1], seqs[b][4][k - 1])
                assert g["n_tracked"] == e.n_tracked and g["align_iters"] == e.align_iters
                assert (g["n_matched"], g["n_reproj_trials"], g["n_pose_obs"]) == (e.n_matched, e.n_reproj_trials, e.n_pose_obs)
                assert g["n_matched"] == 41
                okb = ok[b * N:(b + 1) * N]
                assert np.array_equal(okb, oke) and np.abs(px[b * N:(b + 1) * N][okb == 1] - pxe[oke == 1]).max() <= 1e-3
                rot, trans = synth.pose_error(g["T_cur_w"], np.array(e.T_cur_w[:]))
                assert rot < 1e-9 and trans < 1e-9
                for key in ("n_seeds_updated", "n_seeds_converged", "n_seeds_failed", "n_seeds_skipped"):
                    assert g[key] == getattr(p, key), key
                par.check(seeds_g[b * S:(b + 1) * S], obs_g[b * S:(b + 1) * S], free[b], pinned[b])
        par.finish()
    finally:
        trk.close()
        for s in free + pinned:
            s.close()


# ---------------------------------------------------------------- keyframe insertion (DepthFilter::addKeyframe -> initializeSeeds)
KF_DET = dict(cell=20, levels=3, thr=10.0)


def seed_key_table(px, level, kf, state):
    """alive seeds as sortable rows (kf, level, x, y) + their order"""
    alive = state == 0
    rows = np.stack([kf[alive], level[alive], px[alive, 0].astype(np.int64), px[alive, 1].astype(np.int64)], 1)
    order = np.lexsort(rows.T[::-1])
    return rows[order], np.nonzero(alive)[0][order]


def test_oracle_keyframe_insertion_matches_reference(oracle, ref):
    """Keyframes inserted every third frame: the restatement's add_keyframe (occupancy from the frame's matched features, FAST +
    Shi-Tomasi + grid, one seed per new corner, batch ids, the ageing rule, the ring dropping its oldest keyframe) against the
    reference's own DepthFilter::addKeyframe / removeKeyframe with its FastDetector.  Seed lists: same members, same bits."""
    n_frames = 16
    cfg, poses, imgs, kf, last_px = make_sequence(oracle, "C2", 0x00C0FFEE + 7, n_frames + 1)
    cam = scenes.cam_of(cfg, Cam)
    args = (cam, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"], 100.0, 2.4, 1.2, 3)
    so, sr = OracleSeq(oracle, *args), RefSeq(ref, *args)
    try:
        so.set_pool(3, 2, 3); so.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
        sr.set_pool(3, 2, 3, KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
        S0 = 200
        for s in (so, sr):
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"][:S0], kf["seed_level"][:S0])
            s.set_last(imgs[0])
        n_kf = 0
        for k in range(1, n_frames + 1):
            a, pxa, oka = so.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            b, pxb, okb = sr.step(imgs[k], poses[k - 1], last_px[k - 1], want_px=True)
            assert np.array_equal(np.array(a.T_cur_w[:]), np.array(b.T_cur_w[:])) and a.n_matched == b.n_matched
            # map points are matched against the closest-view observation among the keyframes they were seen in
            assert np.array_equal(oka, okb) and np.array_equal(pxa, pxb), "refined pixels differ at frame %d" % k
            assert a.n_seeds_converged == b.n_seeds_converged and a.n_matched > 80
            if k % 3 == 0:
                na, nb = so.add_keyframe(2.0 + 0.01 * k, 1.0), sr.add_keyframe(2.0 + 0.01 * k, 1.0)
                assert na == nb and na > 50, (na, nb)
                n_kf += 1
            px, lv, kfi, bt, st = so.seed_refs()
            rows_o, idx_o = seed_key_table(px, lv, kfi, st)
            rpx, rlv, rkf, rbt, rst = sr.seed_list()
            rows_r, idx_r = seed_key_table(rpx, rlv, rkf, np.zeros(len(rlv), np.int32))
            assert np.array_equal(rows_o, rows_r), "seed list membership differs at frame %d" % k
            assert np.array_equal(so.seeds()[idx_o].view(np.uint32), rst[idx_r].view(np.uint32)), "seed states differ at frame %d" % k
        assert n_kf == 5 and len(rows_o) > 100
        assert len(np.unique(rows_o[:, 0])) >= 2                      # seeds of several keyframes are alive at the end
    finally:
        so.close(); sr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("batch", [2, 70])
def test_tracker_keyframe_insertion_matches_oracle(ctx, oracle, batch, mode):
    """svob200_tracker_add_keyframe (detect -> seed init -> update, device-resident) against the oracle over a sequence with a
    keyframe every third frame: new-seed counts, pool membership slot by slot, seed bits under the device's pose (pinned oracle)."""
    from android_svo_b200 import capi
    n_frames, n_distinct = 13, min(batch, 2)
    seqs = [make_sequence(oracle, "C2", 0x00C0FFEE + 60 + i, n_frames + 1) for i in range(n_distinct)]
    which = np.arange(batch) % n_distinct
    cfg = seqs[0][0]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    args = (cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    N, S0, CAP = cfg["n_features"], 200, 2400
    pinned = [OracleSeq(oracle, cam_o, *args, 100.0, 2.4, 1.2, 3) for _ in range(n_distinct)]
    trk = capi.Tracker(ctx, cam_g, batch, *args)
    try:
        trk.set_seed_pool(CAP, 3, 2, 3); trk.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
        for s, (_, poses, imgs, kf, _) in zip(pinned, seqs):
            s.set_pool(3, 2, 3); s.set_detector(KF_DET["cell"], KF_DET["levels"], KF_DET["thr"])
            s.set_keyframe(imgs[0], poses[0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"][:S0], kf["seed_level"][:S0])
            s.set_last(imgs[0])
        take = lambda key, n=None: np.concatenate([seqs[w][3][key][:n] for w in which])
        trk.set_keyframe(np.stack([seqs[w][2][0] for w in which]), np.stack([seqs[w][1][0] for w in which]), np.arange(batch + 1) * N,
                         take("kf_px"), take("kf_level"), take("pt_world"), np.arange(batch + 1) * S0, take("seed_px", S0), take("seed_level", S0))
        assert trk.S == batch * CAP
        (trk.set_last if mode == "host" else trk.set_last_device)(np.stack([seqs[w][2][0] for w in which]))
        n_bit_diff = n_seedframes = 0
        for k in range(1, n_frames + 1):
            stats, px_g, ok_g = gpu_step(trk, mode, np.stack([seqs[w][2][k] for w in which]), np.stack([seqs[w][1][k - 1] for w in which]),
                                         np.concatenate([seqs[w][4][k - 1] for w in which]), want_px=True)
            for d in range(n_distinct):
                pinned[d].set_pose_override(stats[d]["T_cur_w"])
                _, px_o, ok_o = pinned[d].step(seqs[d][2][k], seqs[d][1][k - 1], seqs[d][4][k - 1], want_px=True)
                # the closest-view observation of every map point (several keyframes after the first insertion): same choice, same pixels
                for b in np.nonzero(which == d)[0][:3]:
                    assert np.array_equal(ok_g[b * N:(b + 1) * N], ok_o) and np.array_equal(px_g[b * N:(b + 1) * N], px_o), \
                        "map-point matches differ (seq %d, frame %d)" % (b, k)
                assert ok_o.sum() > 80
            if k % 3 == 0:
                n_new, n_drop = trk.add_keyframe(2.0 + 0.01 * k, 1.0)
                assert (n_drop == 0).all()
                for d in range(n_distinct):
                    n_o = pinned[d].add_keyframe(2.0 + 0.01 * k, 1.0)
                    assert (n_new[which == d] == n_o).all(), "new-seed count differs at frame %d: %s vs %d" % (k, n_new[which == d][:4], n_o)
                    assert n_o > 50
            px, lv, kfi, bt, st = trk.seed_refs()
            seeds_g, obs_g = seed_matrix(trk.seeds()), trk.seed_obs()
            for b in range(batch):
                d = which[b]
                opx, olv, okf, obt, ost = pinned[d].seed_refs()
                So = len(olv)
                assert So <= CAP
                sl = slice(b * CAP, b * CAP + So)
                assert np.array_equal(st[sl], ost) and (st[b * CAP + So:(b + 1) * CAP] == 1).all(), "pool occupancy differs (seq %d, frame %d)" % (b, k)
                alive = ost == 0
                assert np.array_equal(px[sl][alive], opx[alive]) and np.array_equal(lv[sl][alive], olv[alive])
                assert np.array_equal(kfi[sl][alive], okf[alive]) and np.array_equal(bt[sl][alive], obt[alive])
                n_bit_diff += int((seeds_g[sl][alive].view(np.uint32) != pinned[d].seeds()[alive].view(np.uint32)).any(axis=1).sum())
                n_seedframes += int(alive.sum())
                oo = pinned[d].seed_obs()
                assert np.array_equal(obs_g["status"][sl], oo["status"]), "seed statuses differ (seq %d, frame %d)" % (b, k)
        print("keyframe insertion: %d seed-frames, %d bit differences under the device's pose" % (n_seedframes, n_bit_diff))
        assert n_bit_diff == 0
        assert len(np.unique(okf[ost == 0])) >= 2
    finally:
        trk.close()
        for s in pinned:
            s.close()
