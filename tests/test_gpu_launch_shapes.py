"""Launch-shape parity: the kernel instances and loop trip counts that launchers pick from the problem's shape, each run at
the shapes that select it and compared with the CPU oracle (oracle/pyoracle.py, oracle/pyoracle_map.py).

- sparse alignment: every instance launch_sparse_align (csrc/sparse_align.cu) can pick — cluster 8 / 4 / 2 and the
  512-, 256- and 128-thread batch kernels — on both sides of every branch, with mixed problem sizes in one launch;
- the pose optimiser beyond one CTA's width (pose_optimize_kernel, POSE_T = 128 threads): strided loops, the outlier
  count across passes, block_median over many and tied values;
- the reprojector's per-image kernel (reproj_cells_kernel) on full-size grids: 1080p at cell 20 (5,184 cells, 21 per
  thread), the 8,192-cell limit and the refusal above it;
- FAST detection (fast_kernel, 120x30 tiles) on levels whose last tile row or column is partial.

Bars as in the rest of the suite: bit-exact where the operation is bit-exact, poses <= 1e-9, discrete outputs equal.
The case-table checks run without a GPU."""
import os
import re
import numpy as np
import pytest

from android_svo_b200 import capi, synth
from oracle.pyoracle import Cam
from oracle import pyoracle_map as pm
import map_scenes as ms
import scenes
from test_gpu_map import check_reproj, to_gpu_records

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ sparse alignment: the launcher's dispatch
def align_instance(batch, max_n):
    """launch_sparse_align (android_svo_b200/csrc/sparse_align.cu) restated: the kernel instance a batch runs on, chosen
    from the batch size and the LARGEST problem of the batch."""
    if batch <= 16 and max_n >= 64:
        return "cluster8"
    if batch <= 32 and max_n >= 64:
        return "cluster4"
    if batch <= 64 and max_n >= 128:
        return "cluster2"
    if max_n > 512:
        return "512"
    if max_n > 128 or batch < 296:
        return "256"
    return "128"


INSTANCES = ("cluster8", "cluster4", "cluster2", "512", "256", "128")
CLUSTER_SIZE = {"cluster8": 8, "cluster4": 4, "cluster2": 2}
# (batch, largest problem, instance)
ALIGN_CASES = [
    (2, 1000, "cluster8"), (16, 64, "cluster8"),
    (17, 64, "cluster4"), (32, 128, "cluster4"),
    (33, 128, "cluster2"), (64, 128, "cluster2"), (64, 1000, "cluster2"),
    (65, 513, "512"), (80, 700, "512"), (70, 1000, "512"),
    (4, 40, "256"), (16, 63, "256"), (33, 127, "256"), (65, 128, "256"), (65, 512, "256"), (295, 128, "256"), (296, 129, "256"),
    (296, 128, "128"),
]
# pairs of cases on the two sides of one branch of the launcher
ALIGN_BOUNDARIES = [((16, 64), (17, 64)), ((32, 128), (33, 128)), ((64, 128), (65, 128)), ((295, 128), (296, 128)),
                    ((16, 63), (16, 64)), ((33, 127), (33, 128)), ((296, 128), (296, 129)), ((65, 512), (65, 513))]
ALIGN_EXTRA_N = (7, 0, 1, 15)        # small problems mixed into every batch (7 and 1 leave CTAs of a cluster without features)
ALIGN_PAIRS = ((0, 3), (1, 4), (2, 6), (0, 1))     # (ref, cur) images of batch slot i: ALIGN_PAIRS[i % 4]
ALIGN_SLOTS = max(b for b, _, _ in ALIGN_CASES)


def align_layout(batch, n):
    """problem size of every batch slot: n everywhere but a few slots (spread over the batch, never slot 0) that hold the
    small problems of ALIGN_EXTRA_N below n"""
    sizes = [n] * batch
    extra = [e for e in ALIGN_EXTRA_N if e < n][:max(batch - 2, 1) if batch > 1 else 0]
    for j, e in enumerate(extra):
        sizes[batch * (j + 1) // (len(extra) + 1)] = e
    return sizes


def test_align_case_table_reaches_every_instance():
    """CPU: the case table reaches all six kernel instances of launch_sparse_align, places both sides of every branch,
    mixes small problems into every batch, and the restated rule still reads like the launcher."""
    src = open(os.path.join(ROOT, "android_svo_b200", "csrc", "sparse_align.cu")).read()
    body = src[src.index("cudaError_t launch_sparse_align("):]
    for line in ("if (batch <= 16 && max_per_problem >= 64) cluster = 8;",
                 "else if (batch <= 32 && max_per_problem >= 64) cluster = 4;",
                 "else if (batch <= 64 && max_per_problem >= 128) cluster = 2;",
                 "if (max_per_problem > 512) sparse_align_kernel<512, 1><<<",
                 "else if (max_per_problem > 128 || batch < 296) sparse_align_kernel<256, 1><<<",
                 "else sparse_align_kernel<128, 1><<<"):
        assert line in body, "launch_sparse_align changed: restate align_instance() and the case table (%s)" % line
    assert len(re.findall(r"sparse_align_kernel<\d+, \d+>", body)) == len(INSTANCES)
    reached = {}
    for batch, n, inst in ALIGN_CASES:
        sizes = align_layout(batch, n)
        assert len(sizes) == batch and max(sizes) == n and sizes[0] == n
        assert align_instance(batch, max(sizes)) == inst, (batch, n)
        assert batch <= ALIGN_SLOTS
        assert {0, 1, 7, 15} & set(sizes) or batch < 2
        if inst in CLUSTER_SIZE:
            assert min(s for s in sizes if s > 0) < CLUSTER_SIZE[inst], "no CTA of the cluster is left without features"
        reached.setdefault(inst, []).append((batch, n))
    assert set(reached) == set(INSTANCES), reached
    assert {(b, n) for b, n, _ in ALIGN_CASES if _ == "512"} >= {(65, 513), (80, 700), (70, 1000)}
    assert (4, 40, "256") in ALIGN_CASES
    table = {(b, n): inst for b, n, inst in ALIGN_CASES}
    for lo, hi in ALIGN_BOUNDARIES:
        assert lo in table and hi in table and table[lo] != table[hi], (lo, hi)


_align_cache = {}


def _align_problem(oracle, k, n):
    """problem of slot kind k (0..3) with n features, and the oracle's result.  Even kinds follow the parity tests'
    layout (features at the image border, one without a point); odd kinds put a third of the features in the bands where
    the coarse levels' 3-px border test flips as the pose moves (the H_ re-use / re-summation test's layout)."""
    key = (k, n)
    if key in _align_cache:
        return _align_cache[key]
    cfg, poses, imgs = scenes.scene("C2", n_frames=8, stride=2, amp=1.0)
    cam_o = scenes.cam_of(cfg, Cam)
    w, h = cfg["w"], cfg["h"]
    a, b = ALIGN_PAIRS[k]
    rng = np.random.RandomState(1000 * k + n)
    has = np.ones(n, np.uint8)
    if n < 8:
        px = np.c_[rng.uniform(60, w - 60, n), rng.uniform(60, h - 60, n)]
    elif k % 2 == 0:
        px = np.c_[rng.uniform(20, w - 20, n), rng.uniform(20, h - 20, n)]
        px[:6] = [[2, 2], [w - 2, h - 2], [5, h / 2], [w - 5, h / 2], [47, 47], [24, 24]]
        has[7] = 0
    else:
        px = np.c_[rng.uniform(60, w - 60, n), rng.uniform(60, h - 60, n)]
        q = n // 3
        px[:2 * q, 0] = np.r_[rng.uniform(40, 58, q), rng.uniform(w - 58, w - 40, q)]
        px[2 * q:2 * q + q // 2, 1] = rng.uniform(40, 58, q // 2)
    ref_pos = oracle.se3_inverse(poses[a])[:3]
    xyz = np.zeros((n, 3))
    for i in range(n):
        _, p = scenes.gt_depth(cfg, poses[a], px[i])
        xyz[i] = oracle.cam2world(cam_o, px[i][0], px[i][1]) * np.sqrt(((p - ref_pos) ** 2).sum())
    T_init = oracle.se3_mul(poses[a], oracle.se3_inverse(poses[a]))
    _, res = oracle.sparse_align(oracle.pyramid(imgs[a], 5), oracle.pyramid(imgs[b], 5), cam_o, px.reshape(-1), xyz.reshape(-1), has, T_init, 4, 2)
    _align_cache[key] = prob = dict(px=px.reshape(-1, 2), has=has, xyz=xyz, T=T_init, res=res)
    return prob


@pytest.fixture(scope="module")
def align_frames(ctx):
    """ALIGN_SLOTS-image reference and current frames; slot i holds the pair ALIGN_PAIRS[i % 4] (a launch of batch B uses
    the first B images)"""
    cfg, poses, imgs = scenes.scene("C2", n_frames=8, stride=2, amp=1.0)
    rid, cid = 9101, 9102
    for fid, side in ((rid, 0), (cid, 1)):
        ctx.frame_create(fid, ALIGN_SLOTS, cfg["w"], cfg["h"], 5)
        ctx.frame_upload(fid, np.stack([imgs[ALIGN_PAIRS[i % 4][side]] for i in range(ALIGN_SLOTS)]))
    yield rid, cid
    ctx.frame_release(rid)
    ctx.frame_release(cid)


@pytest.mark.gpu
@pytest.mark.parametrize("batch,n,inst", ALIGN_CASES, ids=["b%d-n%d-%s" % c for c in ALIGN_CASES])
def test_sparse_align_every_instance(ctx, oracle, align_frames, batch, n, inst):
    """One launch per case: the batch's largest problem picks the instance for every problem of the batch, small
    problems (N = 0, 1, 7, 15) ride along.  Per problem: iterations per level, n_meas, stop, pose < 1e-9, H_ to 1e-9,
    levels run <= factorisations <= iterations; replicas of one problem bit-identical.  (The single-feature problem has
    rank-deficient normal equations: only n_meas and finiteness are defined for it.)"""
    cfg = scenes.scene("C2", n_frames=8, stride=2, amp=1.0)[0]
    sizes = align_layout(batch, n)
    assert align_instance(batch, max(sizes)) == inst
    keys = [(i % 4, s) for i, s in enumerate(sizes)]
    probs = [_align_problem(oracle, k, s) for k, s in keys]
    offs = np.concatenate([[0], np.cumsum(sizes)])
    rid, cid = align_frames
    got = ctx.sparse_align(rid, cid, scenes.cam_of(cfg, capi.Camera), offs, np.concatenate([p["px"] for p in probs]),
                           np.concatenate([p["xyz"] for p in probs]), np.concatenate([p["has"] for p in probs]),
                           np.array([p["T"] for p in probs]), 4, 2)
    first, more, fewer = {}, 0, 0
    for i, (key, p) in enumerate(zip(keys, probs)):
        g, res = got[i], p["res"]
        where = "slot %d (N=%d) of %s" % (i, sizes[i], inst)
        assert g["n_meas"] == res.n_meas, where
        if 0 < sizes[i] < 3:
            # one feature's 16 residuals share one projection Jacobian: J J^T has rank 2 (condition ~1e17), so every
            # Gauss-Newton step is set by rounding and neither the reference's path nor the oracle's is reproducible.
            # What is defined: the problem runs, measures what the oracle measures, stays finite and leaves its
            # neighbours in the launch alone (checked on every other slot).
            assert np.isfinite(g["T_cur_ref"]).all() and g["n_factorisations"] <= int(g["iters"].sum()), where
            assert np.linalg.matrix_rank(np.array(res.H[:]).reshape(6, 6)) < 6, where
            continue
        assert list(g["iters"]) == list(res.iters) and g["stop"] == res.stop, (where, list(g["iters"]), list(res.iters))
        if sizes[i] == 0:
            assert np.array_equal(g["T_cur_ref"], p["T"]) and g["n_factorisations"] == 0, where
        else:
            rot, trans = synth.pose_error(g["T_cur_ref"], np.array(res.T_cur_ref[:]))
            assert rot < 1e-9 and trans < 1e-9, (where, rot, trans)
        H = np.array(res.H[:])
        assert np.abs(g["H"] - H).max() <= 1e-9 * np.abs(H).max(), where
        levels_run, total = int((g["iters"] > 0).sum()), int(g["iters"].sum())
        assert levels_run <= g["n_factorisations"] <= total, (where, g["n_factorisations"], list(g["iters"]))
        if sizes[i] > 0:
            more += g["n_factorisations"] > levels_run
            fewer += g["n_factorisations"] < total
        if key in first:
            assert g.tobytes() == got[first[key]].tobytes(), "%s: replicas of one problem must agree bit for bit" % where
        else:
            first[key] = i
    if inst == "512":
        assert more > 0, "no iteration saw the feature set change: the re-summation is not exercised"
        assert fewer > 0, "no iteration re-used H_: the re-use is not exercised"


# ------------------------------------------------------------------ pose optimiser beyond one CTA
@pytest.fixture(scope="module")
def om(oracle):
    return pm.OracleMap(oracle)


def _ocam(cfg):
    return Cam.make(cfg["w"], cfg["h"], cfg["fx"], cfg["fy"], cfg["cx"], cfg["cy"])


def _gcam(cfg):
    return capi.Camera.make(cfg["w"], cfg["h"], cfg["fx"], cfg["fy"], cfg["cx"], cfg["cy"])


def _pose_frames():
    """(name, px, level, pos, T_init) of one batch: sizes on both sides of the CTA width and far beyond it, even and odd
    n, two frames of duplicated features (ties in the median), a frame with ~70 % gross outliers, an empty frame"""
    out = []
    for n, seed in ((1, 21), (2, 22), (127, 23), (128, 24), (129, 25), (256, 26), (300, 27), (1000, 28), (2500, 29)):
        s = ms.pose_opt_scene(seed=seed, n=n)
        out.append(("n%d" % n, s["px"], s["level"], s["pos"], s["T_init"]))
    s = ms.pose_opt_scene(seed=31, n=150)
    for name, idx in (("dup300", np.repeat(np.arange(150), 2)), ("dup257", np.r_[np.repeat(np.arange(128), 2), 5])):
        out.append((name, s["px"][idx], s["level"][idx], s["pos"][idx], s["T_init"]))
    s = ms.pose_opt_scene(seed=30, n=400, outlier_frac=0.7)
    out.append(("outliers400", s["px"], s["level"], s["pos"], s["T_init"]))
    s = ms.pose_opt_scene(seed=32, n=129, outlier_frac=0.6)
    out.append(("outliers129", s["px"], s["level"], s["pos"], s["T_init"]))
    out.insert(5, ("empty", np.zeros((0, 2)), np.zeros(0, np.int32), np.zeros((0, 3)), ms.pose_opt_scene(seed=3)["T_init"]))
    return out


@pytest.mark.gpu
def test_pose_optimizer_beyond_one_cta(ctx, om):
    """svob200_pose_optimize on one batch mixing 1 to 2,500 features per frame against the oracle: pose <= 1e-9, outlier
    flags, num_obs, iterations and roll-back equal, estimated_scale and error_init exactly equal (order statistics)."""
    cfg = ms.SMALL
    cam_o = _ocam(cfg)
    frames = _pose_frames()
    fs = [np.array([om.o.cam2world(cam_o, p[0], p[1]) for p in px]).reshape(-1, 3) for _, px, _, _, _ in frames]
    off = np.concatenate([[0], np.cumsum([len(lv) for _, _, lv, _, _ in frames])])
    T0 = np.stack([T for *_, T in frames])
    T, res, outl = ctx.pose_optimize(_gcam(cfg), off, np.concatenate(fs), np.concatenate([lv for _, _, lv, _, _ in frames]),
                                     np.concatenate([pos for _, _, _, pos, _ in frames]), T0)
    for b, (name, px, lv, pos, T_init) in enumerate(frames):
        if len(lv) == 0:
            assert np.array_equal(T[b], T0[b]) and res[b]["num_obs"] == 0 and res[b]["iters"] == 0, name
            continue
        To, ro, oo = om.pose_optimize(cam_o, fs[b], lv, pos, T_init)
        rot, trans = synth.pose_error(T[b], To)
        assert rot <= 1e-9 and trans <= 1e-9, (name, rot, trans)
        assert np.array_equal(outl[off[b]:off[b + 1]], oo) and res[b]["num_obs"] == ro["num_obs"], name
        assert res[b]["iters"] == ro["iters"] and res[b]["rolled_back"] == ro["rolled_back"], (name, res[b]["iters"], ro["iters"])
        assert res[b]["estimated_scale"] == ro["estimated_scale"] and res[b]["error_init"] == ro["error_init"], name
        assert np.isclose(res[b]["error_final"], ro["error_final"], rtol=1e-9), name
        assert np.allclose(res[b]["A"], ro["A"], rtol=1e-9, atol=1e-9 * np.abs(ro["A"]).max()), name
        assert np.isclose(res[b]["chi2"], ro["chi2"], rtol=1e-9), name
        if name.startswith("outliers"):
            assert oo.sum() > len(lv) // 2, "%s: most features must be outliers" % name


def test_pose_optimizer_large_frames_oracle_matches_reference(om, ref):
    """CPU: the oracle the GPU test compares with, against the real reference at the large and tied frames."""
    rm = pm.RefMap(ref)
    if not rm.available():
        pytest.skip("oracle/_ref/libsvo_ref.so lacks the map harness")
    cfg = ms.SMALL
    cam = _ocam(cfg)
    img = np.zeros((cfg["h"], cfg["w"]), np.uint8)
    for name, px, lv, pos, T_init in _pose_frames():
        if name not in ("n129", "n1000", "dup300", "dup257", "outliers400"):
            continue
        r = rm.pose_optimize(cam, img, px, lv, pos, T_init)
        f = np.array([om.o.cam2world(cam, p[0], p[1]) for p in px])
        T, res, outl = om.pose_optimize(cam, f, lv, pos, T_init)
        assert np.array_equal(T, r["T"]), name
        assert np.array_equal(outl, r["outlier"]) and res["num_obs"] == r["num_obs"], name
        assert np.allclose(res["A"], r["A"], rtol=1e-6, atol=1e-6 * np.abs(r["A"]).max()), name
        assert np.isclose(res["estimated_scale"], r["estimated_scale"], rtol=1e-6), name
        assert np.isclose(res["error_init"], r["error_init"], rtol=1e-9) and np.isclose(res["error_final"], r["error_final"], rtol=1e-6), name


# ------------------------------------------------------------------ reprojector on full-size grids
HD = dict(w=1920, h=1080, fx=1500.0, fy=1500.0, cx=959.5, cy=539.5, n_levels=5, n_pyr=5)
WIDE = dict(w=2048, h=1024, fx=1600.0, fy=1600.0, cx=1023.5, cy=511.5, n_levels=5, n_pyr=5)
REPROJ_T = 256                      # threads of reproj_cells_kernel (csrc/map_ops.cu)
_map_cache = {}


def _map_scene(oracle, cfg, seed, detect_cell, cell):
    """a map of a few hundred points (the keyframes' FAST corners on a coarse grid of `detect_cell`), reprojected on a
    grid of `cell`, with the oracle's insertion order and keyframe pyramids"""
    key = (cfg["w"], cfg["h"], seed, detect_cell, cell)
    if key not in _map_cache:
        sc = ms.build_map_scene(oracle, cfg=cfg, seed=seed, cell=detect_cell)
        sc["cell"] = cell
        order = ms.insertion_order(sc)
        sc["pts"], sc["obs_o"] = ms.reorder(sc, order)
        sc["kf_pyrs"] = [oracle.pyramid(i, cfg["n_levels"]) for i in sc["kf_imgs"]]
        sc["cur_pyr"] = oracle.pyramid(sc["cur_img"], cfg["n_levels"])
        _map_cache[key] = sc
    return _map_cache[key]


def _oracle_reproject(om, oracle, sc, max_fts):
    cfg = sc["cfg"]
    return om.reproject_map(sc["kf_pyrs"], sc["cur_pyr"], _ocam(cfg), sc["T_cur"], sc["pts"], sc["obs_o"], sc["T_kf"], sc["cell"], max_fts,
                            oracle.matcher_opts(cfg["n_pyr"]))


def _gpu_reproject(ctx, scs, max_fts, cam=None, fid0=9200, launched=None):
    """one svob200_reproject_map call over images b = 0.. (scs[b] None: an image without points, frames of scs[0]);
    launched (a list) receives the kernel launches of that call alone"""
    real = [sc for sc in scs if sc is not None]
    cfg = real[0]["cfg"]
    n_kf = len(real[0]["kf_imgs"])
    kf_fids = [fid0 + 1 + k for k in range(n_kf)]
    img_of = [sc if sc is not None else real[0] for sc in scs]
    for k, fid in enumerate(kf_fids):
        ctx.frame_create(fid, len(scs), cfg["w"], cfg["h"], cfg["n_levels"])
        ctx.frame_upload(fid, np.stack([sc["kf_imgs"][k] for sc in img_of]))
    ctx.frame_create(fid0, len(scs), cfg["w"], cfg["h"], cfg["n_levels"])
    ctx.frame_upload(fid0, np.stack([sc["cur_img"] for sc in img_of]))
    gps, gos, Tos, bases, off = [], [], [], [], [0]
    obs_base = 0
    for b, sc in enumerate(scs):
        bases.append(obs_base)
        if sc is None:
            off.append(off[-1])
            continue
        gp, go, To = to_gpu_records(sc["pts"], sc["obs_o"], sc["T_kf"], kf_fids, b, obs_base)
        gps.append(gp); gos.append(go); Tos.append(To)
        obs_base += len(go); off.append(off[-1] + len(gp))
    n0 = ctx.launch_count()
    try:
        got = ctx.reproject_map(fid0, cam or _gcam(cfg), np.stack([sc["T_cur"] for sc in img_of]), off, np.concatenate(gps), np.concatenate(gos),
                                np.concatenate(Tos), real[0]["cell"], max_fts, ctx.matcher_opts(cfg["n_pyr"]))
    finally:
        if launched is not None:
            launched.append(ctx.launch_count() - n0)
        for fid in kf_fids + [fid0]:
            ctx.frame_release(fid)
    return got, off, bases


def _check_images(om, oracle, scs, max_fts, got, off, bases):
    res, winner, stats = got
    for b, sc in enumerate(scs):
        if sc is None:
            assert (winner[b] == -1).all() and stats[b]["n_matches"] == stats[b]["n_trials"] == stats[b]["n_in_frame"] == 0
            continue
        ores, owinner, nm, nt = _oracle_reproject(om, oracle, sc, max_fts)
        w = winner[b].copy()
        w[w >= 0] -= off[b]
        check_reproj((res[off[b]:off[b + 1]], w, stats[b]), (ores, owinner, nm, nt), bases[b])
        assert stats[b]["n_in_frame"] == int((ores["status"] != pm.REPROJ_NOT_IN_FRAME).sum())
        assert stats[b]["n_cells"] == winner.shape[1]


@pytest.mark.gpu
@pytest.mark.parametrize("max_fts", [0, 37, 150, 100000])
def test_reprojector_1080p_grid(ctx, om, oracle, max_fts):
    """1920x1080 at cell 20: 5,184 cells, 21 per thread of the per-image kernel; images with ~240 and ~450 map points and
    one without; the max_fts cut-off inside a thread's chunk of cells (checked on the oracle's uncapped grid) and at 0."""
    scs = [_map_scene(oracle, HD, 5, 100, 20), _map_scene(oracle, HD, 6, 140, 20), None, _map_scene(oracle, HD, 9, 120, 20)]
    n_cells = -(-HD["w"] // 20) * -(-HD["h"] // 20)
    chunk = -(-n_cells // REPROJ_T)
    assert n_cells == 5184 and chunk == 21
    assert max(len(sc["pts"]) for sc in scs if sc is not None) > REPROJ_T
    inside = 0
    for sc in scs:
        if sc is None:
            continue
        matched = np.flatnonzero(_oracle_reproject(om, oracle, sc, 1 << 30)[1] >= 0)      # cells with a winner, no cut-off
        if 0 < max_fts < len(matched):
            inside += (matched[max_fts] + 1) % chunk != 0       # the first cell left unvisited shares a thread with visited ones
    assert inside > 0 or max_fts == 0 or max_fts >= 1000
    got, off, bases = _gpu_reproject(ctx, scs, max_fts)
    _check_images(om, oracle, scs, max_fts, got, off, bases)


@pytest.mark.gpu
def test_reprojector_grid_limit(ctx, om, oracle):
    """A grid of exactly 8,192 cells (2048x1024 at cell 16) is accepted and matches the oracle; one grid row more is
    refused with SVOB200_ERR_UNSUPPORTED before anything is launched."""
    sc = _map_scene(oracle, WIDE, 7, 100, 16)
    assert -(-WIDE["w"] // 16) * -(-WIDE["h"] // 16) == 8192
    for max_fts in (120, 100000):
        got, off, bases = _gpu_reproject(ctx, [sc, None], max_fts)
        assert got[1].shape == (2, 8192)
        _check_images(om, oracle, [sc, None], max_fts, got, off, bases)
    over = capi.Camera.make(WIDE["w"], WIDE["h"] + 1, WIDE["fx"], WIDE["fy"], WIDE["cx"], WIDE["cy"])    # 128 x 65 = 8,320 cells
    launched = []
    with pytest.raises(capi.Svob200Error, match=r"error -4\b.*8320 cells exceeds the limit of 8192"):
        _gpu_reproject(ctx, [sc], 120, cam=over, launched=launched)
    assert launched == [0], "the refused call launched kernels"


# ------------------------------------------------------------------ FAST detection on partial tiles
FAST_TILE_W, FAST_TILE_H = 120, 30  # fast_kernel's tile (csrc/fast.cu)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,n_levels,cell,thr", [((1080, 1920), 5, 40, 10.0), ((250, 333), 4, 20, 10.0), ((66, 130), 3, 10, 8.0)])
def test_fast_detect_partial_tiles(ctx, oracle, shape, n_levels, cell, thr):
    """svob200_fast_detect where detect levels end in a partial tile row or column (1080p levels 3 and 4 have 135 and 67
    rows), a rendered and a noise image, with and without an occupancy mask: counts, x, y, level and the Shi-Tomasi
    score bits equal to the oracle's."""
    h, w = shape
    cfg = dict(w=w, h=h, fx=0.8 * w, fy=0.8 * w, cx=(w - 1) / 2.0, cy=(h - 1) / 2.0)
    batch = [synth.render(scenes.texture(1024), cfg, synth.trajectory(8, amp_scale=1.0)[3]), scenes.noise_image(h, w, 11)]
    assert any((h >> l) % FAST_TILE_H or (w >> l) % FAST_TILE_W for l in range(n_levels))
    n_cells = -(-w // cell) * -(-h // cell)
    occ = (np.random.RandomState(1).rand(len(batch), n_cells) < 0.2).astype(np.uint8)
    fid = 9300
    ctx.frame_create(fid, len(batch), w, h, n_levels)
    ctx.frame_upload(fid, np.stack(batch))
    in_partial = 0
    try:
        for use_occ in (False, True):
            cells, counts = ctx.fast_detect(fid, n_levels, cell, thr, occ if use_occ else None)
            for b, img in enumerate(batch):
                n, oc = oracle.fast_detect(oracle.pyramid(img, n_levels), n_levels, cell, thr, occ[b] if use_occ else None)
                assert counts[b] == n, (use_occ, b)
                for k in ("x", "y", "level"):
                    assert np.array_equal(cells[b][k], oc[k]), (k, use_occ, b)
                assert np.array_equal(cells[b]["score"].view(np.uint32), oc["score"].view(np.uint32)), "Shi-Tomasi scores differ"
                lv = np.maximum(oc["level"], 0)
                hl, wl = h >> lv, w >> lv
                yl, xl = oc["y"] >> lv, oc["x"] >> lv
                in_partial += int((((yl >= hl // FAST_TILE_H * FAST_TILE_H) | (xl >= wl // FAST_TILE_W * FAST_TILE_W)) & (oc["level"] >= 0)).sum())
    finally:
        ctx.frame_release(fid)
    assert in_partial > 0, "no detected corner lies in a partial tile"
