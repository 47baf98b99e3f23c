"""GPU parity tests: the CUDA path, called through the C ABI (libsvob200.so), against the CPU oracle
on identical seeded inputs.

Bars (north_star): pyramid, FAST corners (+ Shi-Tomasi score, grid selection), warped patches and
ZMSSD bit-exact; poses <= 1e-4 rad / 1e-4 of scene scale (2.0 m); refined pixels <= 1e-3 px; seed
mu/sigma2 relative <= 1e-5.  Discrete decisions (iteration counts, statuses, levels) must be equal.
"""
import ctypes as C
import numpy as np
import pytest

from android_svo_b200 import capi, synth
from oracle.pyoracle import Cam, Seed, SEED_CONVERGED, SEED_NAN_ERASED
import scenes

pytestmark = pytest.mark.gpu

POSE_ROT_TOL = 1e-4          # rad
POSE_TRANS_TOL = 1e-4 * 2.0  # 1e-4 of scene scale (plane at 2 m)
PX_TOL = 1e-3                # px
SEED_REL_TOL = 1e-5

_next_id = [1000]


def new_id():
    _next_id[0] += 1
    return _next_id[0]


def upload(ctx, imgs, n_levels, modes=None):
    """imgs: list of equally sized images -> one frame batch; returns frame id."""
    fid = new_id()
    arr = np.stack(imgs)
    b, h, w = arr.shape
    ctx.frame_create(fid, b, w, h, n_levels)
    ctx.frame_upload(fid, arr, stride=w, round_modes=modes)
    return fid


# ------------------------------------------------------------------ pyramid
@pytest.mark.parametrize("shape,n_levels", [((480, 640), 4), ((480, 640), 5), ((480, 752), 5), ((1080, 1920), 5),
                                            ((60, 94), 3), ((66, 130), 4), ((7, 9), 2), ((64, 64), 7)])
@pytest.mark.parametrize("mode", ["x86", "trunc", "sse2"])
def test_pyramid_bit_exact(ctx, oracle, shape, n_levels, mode):
    h, w = shape
    imgs = [scenes.noise_image(h, w, s, blur=(s % 2 == 0)) for s in range(3)]
    modes = None if mode == "x86" else [0 if mode == "trunc" else 1] * (n_levels - 1)
    if mode == "sse2" and any((w >> l) % 2 for l in range(n_levels - 1)):
        pytest.skip("SSE2 rounding is only defined for even widths")
    fid = upload(ctx, imgs, n_levels, modes)
    try:
        for b, img in enumerate(imgs):
            po = oracle.pyramid(img, n_levels, modes)
            for l in range(n_levels):
                got = ctx.frame_download(fid, b, l)
                assert got.shape == po[l].shape
                assert np.array_equal(got, po[l]), "pyramid level %d of image %d differs (%d px)" % (l, b, (got != po[l]).sum())
    finally:
        ctx.frame_release(fid)


@pytest.mark.parametrize("shape,n_levels,batch,modes", [((480, 640), 4, 96, None), ((480, 752), 5, 80, None), ((1080, 1920), 5, 64, None),
                                                         ((480, 640), 4, 70, [0, 0, 0]), ((480, 640), 3, 65, [1, 0]), ((66, 144), 4, 64, None),
                                                         ((64, 64), 7, 64, None), ((480, 640), 2, 64, None)])
def test_pyramid_bound_batch_bit_exact(ctx, oracle, shape, n_levels, batch, modes):
    """The fused pyramid kernel on batches of 64+ frames bound from a device buffer (the tracker's device-memory path), against
    the oracle's vk::halfSample (vision.cpp:20-110), every level of a sample of the images, bit for bit: frame sizes with
    partial tiles, 2 to 7 levels, both roundings."""
    h, w = shape
    base = [scenes.noise_image(h, w, s, blur=(s % 2 == 0)) for s in range(4)]
    imgs = np.stack([base[i % 4] if i % 5 else np.roll(base[i % 4], i, axis=1) for i in range(batch)])
    d = ctx.dev_alloc(imgs.nbytes)
    ctx.dev_upload(d, imgs)
    fid = new_id()
    ctx.frame_create(fid, batch, w, h, n_levels)
    try:
        ctx.frame_bind(fid, d, w, round_modes=modes)
        ctx.sync()
        for im in (0, 1, 5, batch // 2, batch - 1):
            po = oracle.pyramid(imgs[im], n_levels, modes)
            for l in range(1, n_levels):
                got = ctx.frame_download(fid, im, l)
                assert np.array_equal(got, po[l]), "%dx%d batch %d image %d level %d: %d px differ" % (w, h, batch, im, l, (got != po[l]).sum())
    finally:
        ctx.frame_release(fid)
        ctx.dev_free(d)


def test_pyramid_odd_width_scalar_walk(ctx, oracle):
    """in.cols odd: the reference's scalar path drifts one pixel per row (vision.cpp:92-109); reproduced."""
    img = scenes.noise_image(30, 47, 5)
    got = ctx.half_sample(img, capi.ROUND_TRUNC)
    assert np.array_equal(got, oracle.half_sample(img, 0))
    fid = upload(ctx, [scenes.noise_image(60, 94, 1)], 4)       # 94 -> 47 -> 23 (odd width halved)
    try:
        po = oracle.pyramid(scenes.noise_image(60, 94, 1), 4)
        for l in range(4):
            assert np.array_equal(ctx.frame_download(fid, 0, l), po[l])
    finally:
        ctx.frame_release(fid)


def test_half_sample_standalone(ctx, oracle):
    img = scenes.noise_image(48, 64, 9)
    for mode in (0, 1):
        assert np.array_equal(ctx.half_sample(img, mode), oracle.half_sample(img, mode))


# ------------------------------------------------------------------ FAST
def test_fast_corners_match_cv_fast(ctx, oracle):
    cfg, poses, imgs = scenes.scene("C2")
    test_imgs = [imgs[0], scenes.noise_image(480, 640, 3)]
    fid = upload(ctx, test_imgs, 4)
    try:
        for b, img in enumerate(test_imgs):
            po = oracle.pyramid(img, 4)
            for level in range(3):
                for nonmax in (True, False):
                    gx, gy, gs = ctx.fast_corners(fid, b, level, 10, nonmax)
                    ox, oy, os_ = oracle.fast(po[level], 10, nonmax)
                    assert len(gx) == len(ox) and len(ox) > 0
                    assert np.array_equal(gx, ox) and np.array_equal(gy, oy) and np.array_equal(gs, os_)
    finally:
        ctx.frame_release(fid)


@pytest.mark.parametrize("name,cell,thr", [("C2", 20, 10.0), ("C2", 40, 20.0), ("C3", 30, 10.0), ("C4", 40, 10.1)])
def test_fast_detect_grid_bit_exact(ctx, oracle, name, cell, thr):
    cfg, poses, imgs = scenes.scene(name, n_frames=2)
    nl = cfg["n_levels"]
    batch = [imgs[0], imgs[1], scenes.noise_image(cfg["h"], cfg["w"], 11)]
    n_cells = -(-cfg["w"] // cell) * -(-cfg["h"] // cell)
    rng = np.random.RandomState(0)
    occ = (rng.rand(len(batch), n_cells) < 0.2).astype(np.uint8)
    fid = upload(ctx, batch, nl)
    try:
        for use_occ in (False, True):
            cells, counts = ctx.fast_detect(fid, 3, cell, thr, occ if use_occ else None)
            for b, img in enumerate(batch):
                po = oracle.pyramid(img, nl)
                n, oc = oracle.fast_detect(po, 3, cell, thr, occ[b] if use_occ else None)
                assert counts[b] == n
                for k in ("x", "y", "level"):
                    assert np.array_equal(cells[b][k], oc[k]), k
                assert np.array_equal(cells[b]["score"].view(np.uint32), oc["score"].view(np.uint32)), "Shi-Tomasi scores differ"
    finally:
        ctx.frame_release(fid)


# ------------------------------------------------------------------ sparse image alignment
def _align_problem(cfg, poses, k0, rng, N):
    px = np.c_[rng.uniform(20, cfg["w"] - 20, N), rng.uniform(20, cfg["h"] - 20, N)]
    px[:6] = [[2, 2], [cfg["w"] - 2, cfg["h"] - 2], [5, cfg["h"] / 2], [cfg["w"] - 5, cfg["h"] / 2], [47, 47], [24, 24]]
    has = np.ones(N, np.uint8)
    has[7] = 0
    return px, has


@pytest.mark.parametrize("batch", [1, 20, 40, 70])
def test_sparse_align_cluster_paths(ctx, oracle, batch):
    """The launcher spreads a problem over a thread-block cluster of 8 / 4 / 2 / 1 CTAs depending on the batch size
    (single-stream latency vs throughput); every path must agree with the oracle (same tolerances, same GN iteration
    counts).  The same problem is replicated `batch` times, plus one different problem at the end."""
    cfg, poses, imgs = scenes.scene("C2", n_frames=8, stride=2, amp=1.0)
    nl = 5
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rng = np.random.RandomState(7)
    probs = []
    for (a, b, N) in ((0, 1, 300), (2, 3, 130)):
        px, has = _align_problem(cfg, poses, a, rng, N)
        ref_pos = oracle.se3_inverse(poses[a])[:3]
        xyz = np.zeros((N, 3))
        for i in range(N):
            _, p = scenes.gt_depth(cfg, poses[a], px[i])
            xyz[i] = oracle.cam2world(cam_o, px[i][0], px[i][1]) * np.sqrt(((p - ref_pos) ** 2).sum())
        T_init = oracle.se3_mul(poses[a], oracle.se3_inverse(poses[a]))
        n, res = oracle.sparse_align(oracle.pyramid(imgs[a], nl), oracle.pyramid(imgs[b], nl), cam_o, px.reshape(-1), xyz.reshape(-1), has, T_init, 4, 2)
        probs.append(dict(a=a, b=b, N=N, px=px, has=has, xyz=xyz, T=T_init, n=n, res=res))
    which = [0] * (batch - 1) + [1] if batch > 1 else [0]
    rid = upload(ctx, [imgs[probs[k]["a"]] for k in which], nl)
    cid = upload(ctx, [imgs[probs[k]["b"]] for k in which], nl)
    try:
        offs = np.concatenate([[0], np.cumsum([probs[k]["N"] for k in which])])
        got = ctx.sparse_align(rid, cid, cam_g, offs, np.concatenate([probs[k]["px"] for k in which]), np.concatenate([probs[k]["xyz"] for k in which]),
                               np.concatenate([probs[k]["has"] for k in which]), np.array([probs[k]["T"] for k in which]), 4, 2)
        for i, k in enumerate(which):
            g, res = got[i], probs[k]["res"]
            assert g["n_meas"] == res.n_meas and list(g["iters"]) == list(res.iters) and g["stop"] == res.stop
            rot, trans = synth.pose_error(g["T_cur_ref"], np.array(res.T_cur_ref[:]))
            assert rot < 1e-9 and trans < 1e-9, (rot, trans)
            assert np.allclose(g["H"], np.array(res.H[:]), rtol=1e-9, atol=1e-9 * np.abs(np.array(res.H[:])).max())
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


@pytest.mark.parametrize("batch,N", [(4, 240), (80, 240), (300, 120)])
def test_sparse_align_hessian_reuse_follows_the_feature_set(ctx, oracle, batch, N):
    """An iteration re-uses H_ and its LDLT factor when the set of features inside the current image equals the previous
    iteration's (sparse_align.cu; the reference re-adds the same J J^T every iteration, sparse_img_align.cpp:253-262) and sums /
    factorises again when it does not.  Features are placed in the bands where the 3-px border test of the coarse levels flips as
    the pose moves, so BOTH cases occur; iteration counts, n_meas, H_ and the pose must match the oracle on the cluster kernel
    (batch 4), the 256-thread kernel (batch 80) and the 128-thread batch kernel (batch 300)."""
    cfg, poses, imgs = scenes.scene("C2", n_frames=8, stride=2, amp=1.0)
    nl = 5
    w, h = cfg["w"], cfg["h"]
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rng = np.random.RandomState(3)
    probs = []
    for (a, b) in ((0, 3), (1, 4), (2, 6), (0, 1)):
        px = np.c_[rng.uniform(60, w - 60, N), rng.uniform(60, h - 60, N)]
        k = N // 3
        px[:2 * k, 0] = np.r_[rng.uniform(40, 58, k), rng.uniform(w - 58, w - 40, k)]
        px[2 * k:2 * k + k // 2, 1] = rng.uniform(40, 58, k // 2)
        has = np.ones(N, np.uint8)
        ref_pos = oracle.se3_inverse(poses[a])[:3]
        xyz = np.zeros((N, 3))
        for i in range(N):
            _, p = scenes.gt_depth(cfg, poses[a], px[i])
            xyz[i] = oracle.cam2world(cam_o, px[i][0], px[i][1]) * np.sqrt(((p - ref_pos) ** 2).sum())
        T_init = oracle.se3_mul(poses[a], oracle.se3_inverse(poses[a]))
        n, res = oracle.sparse_align(oracle.pyramid(imgs[a], nl), oracle.pyramid(imgs[b], nl), cam_o, px.reshape(-1), xyz.reshape(-1), has, T_init, 4, 2)
        probs.append(dict(a=a, b=b, px=px, has=has, xyz=xyz, T=T_init, n=n, res=res))
    which = [i % 4 for i in range(batch)]
    rid = upload(ctx, [imgs[probs[k]["a"]] for k in which], nl)
    cid = upload(ctx, [imgs[probs[k]["b"]] for k in which], nl)
    try:
        offs = np.arange(batch + 1) * N
        got = ctx.sparse_align(rid, cid, cam_g, offs, np.concatenate([probs[k]["px"] for k in which]), np.concatenate([probs[k]["xyz"] for k in which]),
                               np.concatenate([probs[k]["has"] for k in which]), np.array([probs[k]["T"] for k in which]), 4, 2)
        more, fewer = 0, 0
        for i, k in enumerate(which):
            g, res = got[i], probs[k]["res"]
            assert g["n_meas"] == res.n_meas and list(g["iters"]) == list(res.iters) and g["stop"] == res.stop, (i, g["iters"], list(res.iters))
            rot, trans = synth.pose_error(g["T_cur_ref"], np.array(res.T_cur_ref[:]))
            assert rot < 1e-9 and trans < 1e-9, (rot, trans)
            H = np.array(res.H[:])
            assert np.abs(g["H"] - H).max() <= 1e-9 * np.abs(H).max()
            levels_run, total = int((g["iters"] > 0).sum()), int(g["iters"].sum())
            assert levels_run <= g["n_factorisations"] <= total, (g["n_factorisations"], g["iters"])
            more += g["n_factorisations"] > levels_run
            fewer += g["n_factorisations"] < total
            if i >= 4:
                assert g.tobytes() == got[i - 4].tobytes(), "replicas of one problem must agree bit for bit"
        assert more > 0, "no iteration saw the feature set change: the test does not exercise the re-summation"
        assert fewer > 0, "no iteration re-used H_: the test does not exercise the re-use"
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


@pytest.mark.parametrize("name,max_level,min_level", [("C2", 3, 2), ("C2", 4, 2), ("C3", 4, 2), ("C2", 2, 0)])
def test_sparse_align_matches_oracle(ctx, oracle, name, max_level, min_level):
    cfg, poses, imgs = scenes.scene(name, n_frames=8, stride=2, amp=1.0)
    nl = 5
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rng = np.random.RandomState(42)
    pairs = [(0, 1), (1, 2), (2, 4), (3, 4), (5, 6)]
    sizes = [120, 300, 16, 0, 700]
    ref_imgs = [imgs[a] for a, _ in pairs]
    cur_imgs = [imgs[b] for _, b in pairs]
    rid, cid = upload(ctx, ref_imgs, nl), upload(ctx, cur_imgs, nl)
    try:
        offs, pxs, xyzs, hass, Ts, exp = [0], [], [], [], [], []
        for (a, b), N in zip(pairs, sizes):
            T_init = oracle.se3_mul(poses[a], oracle.se3_inverse(poses[a]))       # cur starts at the ref pose
            if N:
                px, has = _align_problem(cfg, poses, a, rng, N)
                ref_pos = oracle.se3_inverse(poses[a])[:3]
                xyz = np.zeros((N, 3))
                for i in range(N):
                    _, p = scenes.gt_depth(cfg, poses[a], px[i])
                    f = oracle.cam2world(cam_o, px[i][0], px[i][1])
                    xyz[i] = f * np.sqrt(((p - ref_pos) ** 2).sum())
            else:
                px, has, xyz = np.zeros((0, 2)), np.zeros(0, np.uint8), np.zeros((0, 3))
            pr, pc = oracle.pyramid(imgs[a], nl), oracle.pyramid(imgs[b], nl)
            n, res = oracle.sparse_align(pr, pc, cam_o, px.reshape(-1), xyz.reshape(-1), has, T_init, max_level, min_level)
            exp.append((n, res))
            offs.append(offs[-1] + N); pxs.append(px); xyzs.append(xyz); hass.append(has); Ts.append(T_init)
        got = ctx.sparse_align(rid, cid, cam_g, offs, np.concatenate(pxs), np.concatenate(xyzs), np.concatenate(hass), np.array(Ts),
                               max_level, min_level)
        for i, (n, res) in enumerate(exp):
            g = got[i]
            assert g["n_meas"] == res.n_meas and g["n_meas"] // 16 == n
            assert list(g["iters"]) == list(res.iters), "GN iteration counts differ (decision flip): %s vs %s" % (g["iters"], list(res.iters))
            assert g["stop"] == res.stop
            if sizes[i] == 0:
                assert np.array_equal(g["T_cur_ref"], Ts[i])
                continue
            rot, trans = synth.pose_error(g["T_cur_ref"], np.array(res.T_cur_ref[:]))
            assert rot <= POSE_ROT_TOL and trans <= POSE_TRANS_TOL, (rot, trans)
            assert rot < 1e-9 and trans < 1e-9, "expected near bit-level agreement, got %g %g" % (rot, trans)
            assert abs(g["chi2"] - res.chi2) <= 1e-5 * abs(res.chi2)
            H = np.array(res.H[:])
            assert np.abs(g["H"] - H).max() <= 1e-9 * np.abs(H).max()
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


# ------------------------------------------------------------------ feature alignment
def test_align_patches_bit_exact(ctx, oracle):
    cfg, poses, imgs = scenes.scene("C2")
    nl = 5
    fid = upload(ctx, [imgs[1], imgs[2]], nl)
    rng = np.random.RandomState(3)
    try:
        for level in (0, 1, 2):
            src = oracle.pyramid(imgs[0], nl)[level]
            tgt = [oracle.pyramid(imgs[1], nl)[level], oracle.pyramid(imgs[2], nl)[level]]
            H, W = src.shape
            n = 400
            image = rng.randint(0, 2, n)
            pwb, patch, px0 = np.zeros((n, 100), np.uint8), np.zeros((n, 64), np.uint8), np.zeros((n, 2))
            dirs = rng.randn(n, 2).astype(np.float32)
            dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
            for i in range(n):
                x, y = rng.randint(6, W - 6), rng.randint(6, H - 6)
                pwb[i] = src[y - 5:y + 5, x - 5:x + 5].reshape(-1)
                patch[i] = src[y - 4:y + 4, x - 4:x + 4].reshape(-1)
                px0[i] = [x + rng.uniform(-2, 2), y + rng.uniform(-2, 2)]
                if i % 9 == 0:
                    px0[i] = [rng.uniform(0, W), rng.uniform(0, H)]      # may start out of bounds
            conv, px, _ = ctx.align_patches(fid, level, image, pwb, patch, 10, px0)
            conv1, px1, hinv1 = ctx.align_patches(fid, level, image, pwb, patch, 10, px0, dirv=dirs)
            for i in range(n):
                ok, p = oracle.align2d(tgt[image[i]], pwb[i], patch[i], 10, px0[i])
                assert ok == conv[i]
                assert p.tobytes() == px[i].tobytes(), "align2D px differs: %s vs %s" % (p, px[i])
                ok, p, hi = oracle.align1d(tgt[image[i]], dirs[i], pwb[i], patch[i], 10, px0[i])
                assert ok == conv1[i]
                assert p.tobytes() == px1[i].tobytes() and hi == hinv1[i]
    finally:
        ctx.frame_release(fid)


# ------------------------------------------------------------------ matcher
def _feature_refs(oracle, cam_o, ref_fid, px, levels, T_cur_ref, ref_image=0, cur_image=0, types=None, grads=None):
    n = len(px)
    f = capi.make_feature_refs(n)
    for i in range(n):
        f[i]["ref_frame_id"] = ref_fid if np.isscalar(ref_fid) else ref_fid[i]
        f[i]["ref_image"] = ref_image if np.isscalar(ref_image) else ref_image[i]
        f[i]["cur_image"] = cur_image if np.isscalar(cur_image) else cur_image[i]
        f[i]["level"] = levels[i]
        f[i]["type"] = 0 if types is None else types[i]
        f[i]["px"] = px[i]
        f[i]["f"] = oracle.cam2world(cam_o, px[i][0], px[i][1])
        f[i]["grad"] = (1.0, 0.0) if grads is None else grads[i]
        f[i]["T_cur_ref"] = T_cur_ref if np.ndim(T_cur_ref) == 1 else T_cur_ref[i]
    return f


def test_match_direct_matches_oracle(ctx, oracle):
    cfg, poses, imgs = scenes.scene("C2")
    nl = 5
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rid = upload(ctx, [imgs[0], imgs[1]], nl)          # two keyframes in one batch
    cid = upload(ctx, [imgs[6], imgs[8]], nl)
    cur_idx = [6, 8]
    rng = np.random.RandomState(8)
    n = 600
    try:
        levels = rng.randint(0, 3, n)
        ref_image = rng.randint(0, 2, n)
        cur_image = rng.randint(0, 2, n)
        px = np.floor(np.c_[rng.uniform(2, 638, n), rng.uniform(2, 478, n)] / (1 << levels)[:, None]) * (1 << levels)[:, None]
        types = (np.arange(n) % 9 == 0).astype(int)
        grads = np.tile([0.8, -0.6], (n, 1))
        depth = np.zeros(n); px_in = np.zeros((n, 2)); Tcr = np.zeros((n, 7))
        for i in range(n):
            d, p = scenes.gt_depth(cfg, poses[ref_image[i]], px[i])
            depth[i] = d * (1.0 if i % 5 else rng.uniform(0.3, 0.6))          # some far-off depths -> higher search level
            Tcr[i] = oracle.se3_mul(poses[cur_idx[cur_image[i]]], oracle.se3_inverse(poses[ref_image[i]]))
            pc = synth.se3_transform(poses[cur_idx[cur_image[i]]], p)
            px_in[i] = [cfg["fx"] * pc[0] / pc[2] + cfg["cx"] + rng.uniform(-1.5, 1.5), cfg["fy"] * pc[1] / pc[2] + cfg["cy"] + rng.uniform(-1.5, 1.5)]
        ftrs = _feature_refs(oracle, cam_o, rid, px, levels, Tcr, ref_image, cur_image, types, grads)
        opts_g = ctx.matcher_opts(nl)
        got = ctx.match_direct(cid, cam_g, ftrs, depth, px_in, opts_g)
        opts_o = oracle.matcher_opts(nl)
        pyr_ref = [oracle.pyramid(imgs[0], nl), oracle.pyramid(imgs[1], nl)]
        pyr_cur = [oracle.pyramid(imgs[6], nl), oracle.pyramid(imgs[8], nl)]
        n_ok = 0
        for i in range(n):
            fo = oracle.ref_feature(px[i], ftrs[i]["f"], levels[i], types[i], grads[i])
            ok, m = oracle.find_match_direct(pyr_ref[ref_image[i]], pyr_cur[cur_image[i]], cam_o, fo, depth[i], Tcr[i], opts_o, px_in[i])
            g = got[i]
            assert g["success"] == ok
            if m.search_level == 0 and not np.any(np.array(m.A_cur_ref[:])):
                continue                                                        # rejected before the warp (not in frame)
            assert g["search_level"] == m.search_level
            assert np.array_equal(g["patch_with_border"], np.array(m.patch_with_border[:], np.uint8)), "warped patch differs"
            assert np.array_equal(g["patch"], np.array(m.patch[:], np.uint8))
            assert g["A_cur_ref"].tobytes() == np.array(m.A_cur_ref[:]).tobytes()
            assert np.abs(g["px_cur"] - np.array(m.px_cur[:])).max() <= PX_TOL
            assert g["px_cur"].tobytes() == np.array(m.px_cur[:]).tobytes(), "refined px not bit-exact"
            n_ok += ok
        assert n_ok > n // 2
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


def _epi_inputs(cfg, poses, rng, n):
    levels = rng.randint(0, 3, n)
    px = np.floor(np.c_[rng.uniform(12, cfg["w"] - 12, n), rng.uniform(12, cfg["h"] - 12, n)] / (1 << levels)[:, None]) * (1 << levels)[:, None]
    d = np.zeros((n, 3))
    for i in range(n):
        zgt, _ = scenes.gt_depth(cfg, poses[0], px[i])
        mu = 1.0 / (zgt * rng.uniform(0.7, 1.4))
        sig = rng.choice([0.3, 0.1, 0.02, 0.002])
        d[i] = [1 / mu, 1 / (mu + sig), 1 / max(mu - sig, 1e-8)]
    return levels, px, d


@pytest.mark.parametrize("align_1d", [0, 1])
def test_epipolar_match_matches_oracle(ctx, oracle, align_1d):
    cfg, poses, imgs = scenes.scene("C2")
    nl = 5
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rid = upload(ctx, [imgs[0]], nl)
    cid = upload(ctx, [imgs[3], imgs[7]], nl)
    cur_idx = [3, 7]
    rng = np.random.RandomState(21 + align_1d)
    n = 800
    try:
        levels, px, d = _epi_inputs(cfg, poses, rng, n)
        cur_image = rng.randint(0, 2, n)
        types = (np.arange(n) % 11 == 0).astype(int)
        grads = np.tile([0.6, 0.8], (n, 1))
        Tcr = np.array([oracle.se3_mul(poses[cur_idx[c]], oracle.se3_inverse(poses[0])) for c in cur_image])
        ftrs = _feature_refs(oracle, cam_o, rid, px, levels, Tcr, 0, cur_image, types, grads)
        got = ctx.epipolar_match(cid, cam_g, ftrs, d, ctx.matcher_opts(nl, align_1d=align_1d))
        opts_o = oracle.matcher_opts(nl, align_1d=align_1d)
        pr = oracle.pyramid(imgs[0], nl)
        pc = [oracle.pyramid(imgs[3], nl), oracle.pyramid(imgs[7], nl)]
        n_ok = 0
        for i in range(n):
            fo = oracle.ref_feature(px[i], ftrs[i]["f"], levels[i], types[i], grads[i])
            ok, e = oracle.find_epipolar_match(pr, pc[cur_image[i]], cam_o, fo, Tcr[i], d[i][0], d[i][1], d[i][2], opts_o)
            g = got[i]
            assert g["success"] == ok and g["reject"] == e.reject
            if e.reject:
                continue
            assert g["search_level"] == e.search_level
            assert g["A_cur_ref"].tobytes() == np.array(e.A_cur_ref[:]).tobytes()
            assert g["epi_length"] == e.epi_length
            assert np.array_equal(g["patch_with_border"], np.array(e.patch_with_border[:], np.uint8)), "warped patch differs"
            assert g["n_steps"] == e.n_steps
            assert g["zmssd_best"] == e.zmssd_best, "ZMSSD minimum differs"
            assert g["n_evals"] == e.n_evals
            if ok:
                assert np.abs(g["px_cur"] - np.array(e.px_cur[:])).max() <= PX_TOL
                assert g["px_cur"].tobytes() == np.array(e.px_cur[:]).tobytes(), "px_cur not bit-exact"
                assert abs(g["depth"] - e.depth) <= 1e-12 * e.depth
                n_ok += 1
        assert n_ok > n // 3
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


# ------------------------------------------------------------------ depth filter
def test_update_seed_and_tau_match_oracle(ctx, oracle):
    rng = np.random.RandomState(2)
    n = 4000
    seeds = np.zeros(n, capi.seed_dt)
    seeds["a"], seeds["b"] = rng.uniform(5, 30, n), rng.uniform(5, 30, n)
    seeds["mu"], seeds["z_range"], seeds["sigma2"] = rng.uniform(0.2, 1.0, n), rng.uniform(0.5, 2.0, n), rng.uniform(1e-4, 0.1, n)
    seeds["sigma2"][5] = np.nan
    x = rng.uniform(0.2, 1.0, n).astype(np.float32)
    tau2 = rng.uniform(1e-6, 1e-2, n).astype(np.float32)
    got = ctx.update_seed(x, tau2, seeds)
    n_exact = 0
    for i in range(n):
        s = Seed(*[float(seeds[i][k]) for k in ("a", "b", "mu", "z_range", "sigma2")])
        oracle.update_seed(float(x[i]), float(tau2[i]), s)
        for k in ("a", "b", "mu", "z_range", "sigma2"):
            e, g = np.float32(getattr(s, k)), got[i][k]
            if np.isnan(e):
                assert np.isnan(g)
                continue
            assert abs(g - e) <= SEED_REL_TOL * abs(e), (k, g, e)       # exp() is the only libm call on this path
        n_exact += all(np.float32(getattr(s, k)).tobytes() == got[i][k].tobytes() for k in ("a", "b", "mu", "sigma2"))
    assert n_exact > 0.9 * n
    cam_o = Cam.make(640, 480, 525, 525, 319.5, 239.5)
    T = np.array([oracle.se3_exp(rng.randn(6) * [0.2, 0.2, 0.05, 0.02, 0.02, 0.02]) for _ in range(n)])
    f = np.array([oracle.cam2world(cam_o, rng.uniform(0, 640), rng.uniform(0, 480)) for _ in range(n)])
    z = rng.uniform(1, 4, n)
    ang = 2 * np.arctan(1 / (2 * 525.0))
    tau = ctx.compute_tau(T, f, z, ang)
    for i in range(n):
        e = oracle.compute_tau(T[i], f[i], z[i], ang)
        assert abs(tau[i] - e) <= 1e-9 * abs(e)


def test_seeds_update_matches_oracle(ctx, oracle):
    cfg, poses, imgs = scenes.scene("C2")
    nl = 5
    cam_o, cam_g = scenes.cam_of(cfg, Cam), scenes.cam_of(cfg, capi.Camera)
    rid = [upload(ctx, [imgs[0]], nl), upload(ctx, [imgs[1]], nl)]       # two keyframes, separate frames
    rng = np.random.RandomState(5)
    S = 700
    seed_ref = rng.randint(0, 2, S)
    levels = rng.randint(0, 3, S)
    px = np.floor(np.c_[rng.uniform(12, 628, S), rng.uniform(12, 468, S)] / (1 << levels)[:, None]) * (1 << levels)[:, None]
    px[:4] = [[0, 0], [636, 476], [8, 8], [320, 240]]
    seeds = np.zeros(S, capi.seed_dt)
    for i in range(S):
        zgt, _ = scenes.gt_depth(cfg, poses[seed_ref[i]], px[i])
        s = oracle.seed_init(zgt * rng.uniform(0.8, 1.3), zgt * 0.5)
        seeds[i] = (s.a, s.b, s.mu, s.z_range, s.sigma2)
    seeds["sigma2"][9] = np.nan
    pyr = [oracle.pyramid(im, nl) for im in imgs]
    opts_o, opts_g = oracle.matcher_opts(nl), ctx.matcher_opts(nl)
    cids = []
    try:
        total_conv = 0
        for frame in range(2, 10):
            cid = upload(ctx, [imgs[frame]], nl)
            cids.append(cid)
            n = len(px)
            ftrs = _feature_refs(oracle, cam_o, [rid[r] for r in seed_ref], px, levels, np.zeros(7))
            T_ref_w = np.array([poses[r] for r in seed_ref])
            got_seeds, obs = ctx.seeds_update(cid, cam_g, ftrs, T_ref_w, poses[frame][None, :], opts_g, 100.0, seeds)
            exp_seeds = seeds.copy()
            status = np.zeros(n, np.int32)
            for i in range(n):
                s = Seed(*[float(seeds[i][k]) for k in ("a", "b", "mu", "z_range", "sigma2")])
                fo = oracle.ref_feature(px[i], ftrs[i]["f"], levels[i])
                st, epi = oracle.update_seed_with_frame(pyr[seed_ref[i]], pyr[frame], cam_o, fo, poses[seed_ref[i]], poses[frame], opts_o, 100.0, s, want_epi=True)
                status[i] = st
                exp_seeds[i] = (s.a, s.b, s.mu, s.z_range, s.sigma2)
                assert obs[i]["status"] == st, "seed %d: status %d vs %d" % (i, obs[i]["status"], st)
                if st >= 3:
                    assert obs[i]["zmssd_best"] == epi.zmssd_best and obs[i]["n_evals"] == epi.n_evals
                if st >= 4:
                    assert abs(obs[i]["z"] - epi.depth) <= 1e-12 * epi.depth
                    assert np.abs(obs[i]["px_cur"] - np.array(epi.px_cur[:])).max() <= PX_TOL
            for k in ("a", "b", "mu", "z_range", "sigma2"):
                e, g = exp_seeds[k], got_seeds[k]
                both_nan = np.isnan(e) & np.isnan(g)
                assert np.all(both_nan | (np.abs(g - e) <= SEED_REL_TOL * np.abs(e))), k
            total_conv += int((status == SEED_CONVERGED).sum())
            keep = (status != SEED_CONVERGED) & (status != SEED_NAN_ERASED)
            seeds, px, levels, seed_ref = exp_seeds[keep], px[keep], levels[keep], seed_ref[keep]
        assert total_conv > S // 3
    finally:
        for f in rid + cids:
            ctx.frame_release(f)


# ------------------------------------------------------------------ full-size properties
def test_full_size_pyramid_properties(ctx, oracle):
    """C4-size batch: level l+1 of the device pyramid equals half-sampling the downloaded level l
    (checksum of all levels against the oracle applied level by level)."""
    cfg = synth.CONFIGS["C4"]
    imgs = [scenes.noise_image(cfg["h"], cfg["w"], s) for s in range(4)]
    fid = upload(ctx, imgs, 5)
    try:
        for b in range(4):
            prev = ctx.frame_download(fid, b, 0)
            assert np.array_equal(prev, imgs[b])
            for l in range(1, 5):
                cur = ctx.frame_download(fid, b, l)
                assert np.array_equal(cur, oracle.half_sample(prev, oracle.lib.svo_oracle_half_sample_mode_x86(prev.shape[1])))
                prev = cur
    finally:
        ctx.frame_release(fid)


# ------------------------------------------------------------------ exact float chi2 chain (sparse alignment's rollback test)
def _chain_cases():
    """(name, residuals [N,16] float32, visible, contrib): realistic residuals plus inputs built to hit every special case of
    the parallel replay — exact ties (the term is half an ulp of the running sum), binade crossings in late chunks, zeros,
    skipped features, terms far larger than the sum, sums that stay tiny, overflow to infinity."""
    rng = np.random.default_rng(77)
    cases = []
    for n in (1, 7, 120, 128, 129, 300, 1000, 2048, 3001):
        res = (rng.standard_normal((n, 16)) * rng.choice([0.5, 8.0, 40.0])).astype(np.float32)
        cases.append(("gauss%d" % n, res, np.ones(n, np.uint8), (rng.random(n) > 0.1).astype(np.uint8)))
    # dyadic residuals: squares are exact small multiples of powers of two => exact ties as soon as the sum's ulp doubles past them
    for n, lo in ((1000, -6), (2048, -9), (777, -3)):
        e = rng.integers(lo, 4, size=(n, 16))
        m = rng.choice([1.0, 1.5, 3.0, 0.75, 1.25], size=(n, 16))
        res = (m * np.exp2(e)).astype(np.float32) * rng.choice([-1.0, 1.0], size=(n, 16)).astype(np.float32)
        cases.append(("dyadic%d_%d" % (n, lo), res, np.ones(n, np.uint8), np.ones(n, np.uint8)))
    # saturated residuals (|res| = 255): the sum crosses 2^27, 2^28, ... in the parallel chunks
    res = np.full((3000, 16), 255.0, np.float32)
    res[::7] = 254.5
    cases.append(("saturated", res, np.ones(3000, np.uint8), np.ones(3000, np.uint8)))
    # mostly zeros with a few spikes; features switched off by either flag
    res = np.zeros((1500, 16), np.float32)
    res[rng.integers(0, 1500, 40), rng.integers(0, 16, 40)] = (rng.standard_normal(40) * 100).astype(np.float32)
    cases.append(("sparse", res, (rng.random(1500) > 0.3).astype(np.uint8), (rng.random(1500) > 0.3).astype(np.uint8)))
    cases.append(("allzero", np.zeros((600, 16), np.float32), np.ones(600, np.uint8), np.ones(600, np.uint8)))
    cases.append(("alloff", np.ones((600, 16), np.float32), np.zeros(600, np.uint8), np.ones(600, np.uint8)))
    # first chunk zero, the rest not: the parallel chunks start from s = 0
    res = (rng.standard_normal((900, 16)) * 10).astype(np.float32)
    res[:128] = 0
    cases.append(("zerohead", res, np.ones(900, np.uint8), np.ones(900, np.uint8)))
    # terms far larger than the running sum, in late chunks
    res = (rng.standard_normal((1200, 16)) * 3).astype(np.float32)
    res[500, 3] = 1e10
    res[900, 9] = 3e15
    res[1100, 0] = 1e19
    cases.append(("huge", res, np.ones(1200, np.uint8), np.ones(1200, np.uint8)))
    res = (rng.standard_normal((700, 16)) * 3).astype(np.float32)
    res[400, 5] = 3e19                                  # the square overflows float
    cases.append(("inf", res, np.ones(700, np.uint8), np.ones(700, np.uint8)))
    # sums that stay below 2^-95 (the parallel path hands over to the sequential one) and denormal squares
    cases.append(("tiny", (rng.standard_normal((500, 16)) * 1e-17).astype(np.float32), np.ones(500, np.uint8), np.ones(500, np.uint8)))
    cases.append(("denormal", (rng.standard_normal((500, 16)) * 1e-21).astype(np.float32), np.ones(500, np.uint8), np.ones(500, np.uint8)))
    # a tiny head then ordinary terms: the sum climbs through a hundred binades inside a parallel chunk
    res = (rng.standard_normal((640, 16)) * 1e-12).astype(np.float32)
    res[300:] = (rng.standard_normal((340, 16)) * 5).astype(np.float32)
    cases.append(("climb", res, np.ones(640, np.uint8), np.ones(640, np.uint8)))
    # every term a tie candidate: sum sits at 2^24-ish with ulp 2, terms 1.0 (half an ulp) and 3.0
    res = np.ones((2000, 16), np.float32)
    res[:128] = 362.0                                   # first chunk lifts the sum to 2048 * 131044 ~ 2^28
    res[128:, ::2] = np.float32(np.sqrt(8.0))           # not exact: ordinary terms in between
    res[128:, 1::4] = 4.0                               # 16 = half an ulp of [2^28, 2^29) => ties
    cases.append(("ties", res, np.ones(2000, np.uint8), np.ones(2000, np.uint8)))
    return cases


def _chain_reference(res, visible, contrib):
    """The reference's `float chi2; chi2 += res*res*weight` (sparse_img_align.cpp:259-263) over the contributing features."""
    on = (visible != 0) & (contrib != 0)
    with np.errstate(over="ignore", invalid="ignore"):
        t = (res[on] * res[on]).astype(np.float32).ravel()
        if t.size == 0:
            return np.float32(0), 0
        return np.cumsum(t, dtype=np.float32)[-1], int(t.size)    # cumsum accumulates sequentially in float32


@pytest.mark.parametrize("block", [128, 256, 512])
def test_exact_chi2_chain_parallel_property(ctx, block):
    for name, res, vis, con in _chain_cases():
        want, want_n = _chain_reference(res, vis, con)
        bits = lambda v: int(np.float32(v).view(np.uint32))
        for which, (got, got_n) in zip(("serial", "parallel/latency", "parallel/batch"), ctx.debug_chi2_chain(res, vis, con, block=block)):
            assert got_n == want_n, (name, which, got_n, want_n)
            assert bits(got) == bits(want), "%s: %s device chain %r (%08x) != reference %r (%08x)" % (name, which, got, bits(got), want, bits(want))
