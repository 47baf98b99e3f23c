"""GPU: the C-ABI entry points the C++ drop-in (android_svo_b200/host/svo_b200_dropin.cpp) calls, called the way it calls them.

tests/test_dropin.py runs the drop-in itself inside the reference's own control flow; that needs the original Android SVO
sources and skips without them.  These tests need nothing outside the repository.  They cover the entry points only the
drop-in uses: svob200_shi_tomasi, svob200_warp_matrix_affine, svob200_warp_affine, svob200_depth_from_triangulation,
svob200_frame_upload_level and the stand-alone svob200_half_sample.  They also cover two contexts driven from two host
threads, the drop-in's two-thread layout.  Each result is checked against the reference's outputs stored in
tests/golden/reference_golden.npz where those exist, and against the C restatement (oracle/), pinned to the same
outputs by tests/test_oracle_golden.py.
"""
import ctypes as C
import os
import threading
import numpy as np
import pytest

from android_svo_b200 import capi
from oracle.pyoracle import Cam
import scenes
from test_pipeline import make_sequence

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz"))
P = capi._ptr


def u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def golden_cam(cls):
    c = G["scene_cam"]
    return cls.make(int(c[0]), int(c[1]), *c[2:])


# ---------------------------------------------------------------- thin wrappers, one item layout as the drop-in passes it
def shi_tomasi(ctx, img, uv):
    img, uv = u8(img), np.ascontiguousarray(uv, dtype=np.int32).reshape(-1, 2)
    out = np.zeros(len(uv), np.float32)
    ctx._ck(ctx.L.svob200_shi_tomasi(ctx.h, P(img), img.shape[1], img.shape[0], img.shape[1], len(uv), P(uv), P(out)))
    return out


def warp_matrix_affine(ctx, cam, px, f, depth, T_cur_ref, level):
    px, f, depth, T = f64(px).reshape(-1, 2), f64(f).reshape(-1, 3), f64(depth).reshape(-1), f64(T_cur_ref).reshape(-1, 7)
    level = np.ascontiguousarray(level, dtype=np.int32).reshape(-1)
    A = np.zeros((len(px), 4))
    ctx._ck(ctx.L.svob200_warp_matrix_affine(ctx.h, C.byref(cam), len(px), P(px), P(f), P(depth), P(T), P(level), P(A), capi.MEM_HOST))
    return A


def warp_affine(ctx, img, A, px, level_ref, search_level, patch):
    img, A, px = u8(img), f64(A), f64(px)
    ctx._ck(ctx.L.svob200_warp_affine(ctx.h, P(img), img.shape[1], img.shape[0], img.shape[1], P(A), P(px), int(level_ref),
                                      int(search_level), 5, P(patch)))
    return patch


def depth_from_triangulation(ctx, T_search_ref, f_ref, f_cur, depth):
    T, a, b = f64(T_search_ref).reshape(-1, 7), f64(f_ref).reshape(-1, 3), f64(f_cur).reshape(-1, 3)
    depth = f64(depth).copy()
    ok = np.zeros(len(T), np.int32)
    ctx._ck(ctx.L.svob200_depth_from_triangulation(ctx.h, len(T), P(T), P(a), P(b), P(depth), P(ok)))
    return depth, ok


def oracle_depth_from_triangulation(oracle, T, a, b, depth):
    d = C.c_double(depth)
    T, a, b = f64(T), f64(a), f64(b)
    ok = oracle.lib.svo_oracle_depth_from_triangulation(P(T), P(a), P(b), C.byref(d))
    return d.value, int(ok)


def epi_T_cur_ref(oracle):
    poses = G["scene_poses"]
    return np.array([oracle.se3_mul(poses[int(c)], oracle.se3_inverse(poses[0])) for c in G["epi_cur"]])


# ---------------------------------------------------------------- vk::shiTomasiScore
def test_shi_tomasi_vs_reference_golden(ctx):
    got = shi_tomasi(ctx, G["st_img"], G["st_uv"])
    assert got.view(np.uint32).tobytes() == G["st_score"].view(np.uint32).tobytes()


@pytest.mark.parametrize("source", ["scene", "noise"])
def test_shi_tomasi_matches_oracle(ctx, oracle, source):
    img = scenes.scene("C2", 3)[2][0] if source == "scene" else scenes.noise_image(480, 640, 4)
    rng = np.random.RandomState(11)
    uv = np.concatenate([[(100, 100), (5, 5), (320, 240), (634, 474), (635, 100), (17, 333), (0, 0), (639, 479)],
                         np.stack([rng.randint(0, 640, 300), rng.randint(0, 480, 300)], 1)]).astype(np.int32)
    got = shi_tomasi(ctx, img, uv)
    want = np.array([oracle.shi_tomasi(img, u, v) for u, v in uv], np.float32)
    assert got.tobytes() == want.tobytes()


# ---------------------------------------------------------------- warp::getWarpMatrixAffine / warp::warpAffine
def test_warp_matrix_affine_vs_reference_golden(ctx, oracle):
    """A_cur_ref of the reference's findEpipolarMatchDirect (d_estimate, the feature's level), all items in one call and one item
    per call as the drop-in calls it"""
    cam = golden_cam(capi.Camera)
    T = epi_T_cur_ref(oracle)
    d = G["epi_d"][:, 0]
    A = warp_matrix_affine(ctx, cam, G["epi_px"], G["epi_f"], d, T, G["epi_level"])
    assert A.tobytes() == G["epi_A"].tobytes()
    for i in range(0, len(d), 7):
        one = warp_matrix_affine(ctx, cam, G["epi_px"][i], G["epi_f"][i], d[i], T[i], G["epi_level"][i])
        assert one.tobytes() == G["epi_A"][i:i + 1].tobytes()


def test_warp_affine_vs_reference_golden(ctx, oracle):
    """patch_with_border of the reference's findEpipolarMatchDirect: the reference's A_cur_ref and search level, the reference
    image's level of the feature"""
    pyr = oracle.pyramid(G["scene_imgs"][0], 4)
    for i in range(len(G["epi_px"])):
        lvl = int(G["epi_level"][i])
        patch = warp_affine(ctx, pyr[lvl], G["epi_A"][i], G["epi_px"][i], lvl, int(G["epi_sl"][i]), np.zeros(100, np.uint8))
        assert np.array_equal(patch, G["epi_pwb"][i]), "item %d" % i


def test_warp_affine_matches_oracle(ctx, oracle):
    """random affine warps on every level, and a NaN warp, which leaves the patch untouched like the reference"""
    cfg, poses, imgs = scenes.scene("C2", 3)
    pyr = oracle.pyramid(imgs[0], cfg["n_levels"])
    rng = np.random.RandomState(3)
    for i in range(200):
        lvl, sl = rng.randint(0, 3), rng.randint(0, 4)
        A = np.eye(2).reshape(-1) + rng.uniform(-0.3, 0.3, 4)
        px = np.array([rng.uniform(-8, 648), rng.uniform(-8, 488)])
        got = warp_affine(ctx, pyr[lvl], A, px, lvl, sl, np.full(100, 77, np.uint8))
        want, img = np.full(100, 77, np.uint8), u8(pyr[lvl])
        oracle.lib.svo_oracle_warp_affine(P(A), P(img), img.shape[1], img.shape[0], P(px), lvl, sl, 5, P(want))
        assert np.array_equal(got, want), "warp %d" % i
    got = warp_affine(ctx, pyr[0], np.full(4, np.nan), np.array([320.0, 240.0]), 0, 0, np.full(100, 77, np.uint8))
    assert (got == 77).all()


# ---------------------------------------------------------------- depthFromTriangulation
def test_depth_from_triangulation_vs_reference_golden(ctx, oracle):
    """the depth of every successful epipolar match of the reference, from T_cur_ref, the feature's bearing and the bearing of the
    reference's matched pixel (to 1e-12 relative, the bar of tests/test_gpu_golden.py::test_epipolar_vs_reference)"""
    cam = golden_cam(Cam)
    ok = G["epi_ok"].astype(bool)
    f_cur = np.array([oracle.cam2world(cam, p[0], p[1]) for p in G["epi_px_cur"][ok]])
    depth, good = depth_from_triangulation(ctx, epi_T_cur_ref(oracle)[ok], G["epi_f"][ok], f_cur, np.zeros(int(ok.sum())))
    assert good.all() and ok.sum() > 50
    assert np.abs(depth - G["epi_depth"][ok]).max() <= 1e-12 * G["epi_depth"][ok].max()


def test_depth_from_triangulation_matches_oracle(ctx, oracle):
    """random geometry plus parallel rays (the reference returns false and leaves depth as it was)"""
    rng = np.random.RandomState(8)
    n = 400
    T = np.array([oracle.se3_exp(rng.randn(6) * [0.3, 0.3, 0.1, 0.05, 0.05, 0.05]) for _ in range(n)])
    a = rng.randn(n, 3); a[:, 2] = np.abs(a[:, 2]) + 0.5; a /= np.linalg.norm(a, axis=1, keepdims=True)
    b = rng.randn(n, 3); b[:, 2] = np.abs(b[:, 2]) + 0.5; b /= np.linalg.norm(b, axis=1, keepdims=True)
    T[:20, 3:] = [0.0, 0.0, 0.0, 1.0]                 # no rotation and b = a: parallel rays
    b[:20] = a[:20]
    d0 = rng.uniform(1, 3, n)
    depth, ok = depth_from_triangulation(ctx, T, a, b, d0)
    for i in range(n):
        want, wok = oracle_depth_from_triangulation(oracle, T[i], a[i], b[i], d0[i])
        assert ok[i] == wok and abs(depth[i] - want) <= 1e-12 * abs(want), "item %d" % i
    assert not ok[:20].any() and np.array_equal(depth[:20], d0[:20]) and ok[20:].sum() > 300


# ---------------------------------------------------------------- svob200_frame_upload_level / svob200_half_sample
@pytest.mark.parametrize("h,w,n_levels", [(480, 640, 4), (60, 94, 3)])
def test_frame_upload_level_mirrors_host_pyramid(ctx, oracle, h, w, n_levels):
    """a host pyramid mirrored level by level is held verbatim (truncating levels, which a rebuild on this width would not make) and
    FAST + Shi-Tomasi + grid on the mirror equals the oracle's on the host pyramid"""
    img = scenes.noise_image(h, w, 21)
    pyr = oracle.pyramid(img, n_levels, [0] * (n_levels - 1))
    fid = 7301
    ctx.frame_create(fid, 1, w, h, n_levels)
    try:
        for l in range(n_levels):
            lv = u8(pyr[l])
            ctx._ck(ctx.L.svob200_frame_upload_level(ctx.h, fid, 0, l, P(lv), lv.shape[1]))
        for l in range(n_levels):
            assert np.array_equal(ctx.frame_download(fid, 0, l), pyr[l]), "level %d" % l
        cells, _ = ctx.fast_detect(fid, n_levels, 20, 10.0)
        _, oc = oracle.fast_detect(pyr, n_levels, 20, 10.0)
        assert np.array_equal(cells[0]["x"], oc["x"]) and np.array_equal(cells[0]["y"], oc["y"]) and np.array_equal(cells[0]["level"], oc["level"])
        assert cells[0]["score"].view(np.uint32).tobytes() == oc["score"].view(np.uint32).tobytes()
    finally:
        ctx.frame_release(fid)


@pytest.mark.parametrize("key", ["sse2", "trunc"])
def test_half_sample_chain_vs_reference_golden(ctx, key):
    """vk::halfSample called level by level on the host image, as createImgPyramid calls it, against the reference's levels; the
    x86 build picks SSE2 where the input width is a multiple of 16"""
    lv = G["pyr_img"]
    for l in range(1, 4):
        mode = ctx.L.svob200_round_mode_x86(lv.shape[1]) if key == "sse2" else capi.ROUND_TRUNC
        lv = ctx.half_sample(lv, mode)
        assert np.array_equal(lv, G["pyr_%s_l%d" % (key, l)]), "level %d" % l


# ---------------------------------------------------------------- two contexts from two host threads
def run_sequence(ctx, seq, mode):
    cfg, poses, imgs, kf, last_px = seq
    cam = scenes.cam_of(cfg, capi.Camera)
    trk = capi.Tracker(ctx, cam, 1, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"])
    try:
        N, S = len(kf["kf_px"]), len(kf["seed_px"])
        trk.set_keyframe(imgs[0][None], poses[0][None], [0, N], kf["kf_px"], kf["kf_level"], kf["pt_world"], [0, S], kf["seed_px"], kf["seed_level"])
        (trk.set_last if mode == "host" else trk.set_last_device)(imgs[0][None])
        out = []
        for k in range(1, len(imgs)):
            st = (trk.step if mode == "host" else trk.step_device)(imgs[k][None], poses[k - 1][None], last_px[k - 1])
            out.append(st.tobytes())
        out.append(trk.seeds().tobytes())
        return out
    finally:
        trk.close()


@pytest.mark.parametrize("mode", ["host", "device"])
def test_two_contexts_from_two_threads(ctx, oracle, mode):
    """the drop-in's two-thread layout serves each thread from its own svob200 context: two sequences tracked at the same time on two
    contexts give the bits they give one after the other on one"""
    seqs = [make_sequence(oracle, "C2", 0x00C0FFEE + 40 + i, 6) for i in range(2)]
    want = [run_sequence(ctx, s, mode) for s in seqs]
    ctx2 = capi.Context(0)
    try:
        got, errors = [None, None], []

        def worker(i, c):
            try:
                got[i] = run_sequence(c, seqs[i], mode)
            except Exception as e:        # surfaced below: a thread's exception does not fail the test by itself
                errors.append(e)
        threads = [threading.Thread(target=worker, args=(0, ctx)), threading.Thread(target=worker, args=(1, ctx2))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors, errors
        assert got == want
    finally:
        ctx2.close()
