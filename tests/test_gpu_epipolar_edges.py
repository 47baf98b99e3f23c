"""Edge cases of the epipolar search (Matcher::findEpipolarMatchDirect, matcher.cpp:207-355) built on purpose, against the
oracle: walks of exact lengths around the 32-sample staging chunks of the search kernel and around the step limit, ZMSSD ties
that the kernel settles by a (score, step) minimum across the 8 lanes of a group, the DIRECT / WALK switch at epi_length 2.0,
segments that cross the image border or reach beyond the short2 pixel range, infinite and NaN depth ranges, edgelet filtering,
every combination of subpix_refinement and align_1d, and step limits above 1,023 and walks above 65,536 samples.  The same
geometry then runs through the depth filter (svob200_seeds_update).

Bars as in test_gpu_parity: success, reject, search_level, n_steps, n_evals and zmssd_best equal; A_cur_ref, epi_length, the
warped patches and px_cur bit-exact; depth within 1e-12 relative."""
import ctypes as C
import functools
import numpy as np
import pytest

from android_svo_b200 import capi
from oracle.pyoracle import Cam, Seed
import scenes
from test_gpu_parity import upload, _feature_refs, PX_TOL, SEED_REL_TOL

NL = 5                                   # pyramid levels: search levels 0 .. 4
INT_MAX = 2 ** 31 - 1
INF_DEPTH = 1.0 / float(np.float32(1e-8))    # d_max of a seed whose z_inv_max is clamped (depth_filter.cpp:328)
ERR_ARG = -1                             # SVOB200_ERR_ARG
SEARCH_CTAS = 5                          # resident CTAs per SM of the persistent search kernel (matcher.cu), 16 groups each
WALK_TARGETS = (2, 31, 32, 33, 63, 64, 65, 999, 1000, 1001)
LIMITS = (1, 32, 1000, 1023, 1024, 1500, 5000, INT_MAX)
LONG_TARGETS = (1023, 1024, 1025, 1500, 1501, 5000, 5001, 65600)
PERIOD = 13                              # px: the current image of the tie cases repeats along x
IDENT = [0.0, 0.0, 0.0, 1.0]
# pure translations (x, y, z, then the identity quaternion): T_SCENE moves sideways with a tiny forward component, so its
# epipole lies ~160,000 px to the right and a segment can be made as long as wanted by lowering d_min
T_SCENE = np.array([0.15, 0.02, 0.0005] + IDENT)
T_X = np.array([0.05, 0.0, 0.0] + IDENT)
T_Y = np.array([0.0, -0.1, 0.0005] + IDENT)


class World:
    """Three reference / current image pairs in one frame batch each: 0 the rendered plane seen from a pose and from T_SCENE
    times that pose (true matches exist), 1 an image periodic along x (both sides), 2 a flat image (both sides)."""

    def __init__(self, oracle):
        cfg, poses, imgs = scenes.scene("C2")
        self.cfg, self.P0 = cfg, poses[0]
        self.cam = scenes.cam_of(cfg, Cam)
        self.P1 = oracle.se3_mul(T_SCENE, poses[0])
        from android_svo_b200 import synth
        cur = synth.render(scenes.texture(), cfg, self.P1)
        periodic = np.tile(scenes.noise_image(cfg["h"], PERIOD, 5), (1, cfg["w"] // PERIOD + 1))[:, :cfg["w"]]
        flat = np.full((cfg["h"], cfg["w"]), 128, np.uint8)
        self.ref_imgs, self.cur_imgs = [imgs[0], periodic, flat], [cur, periodic, flat]
        self.pr = [oracle.pyramid(i, NL) for i in self.ref_imgs]
        self.pc = [oracle.pyramid(i, NL) for i in self.cur_imgs]


@functools.lru_cache(maxsize=None)
def world(oracle):
    return World(oracle)


def _case(name, img, px, level, T, d, ftype=0, grad=(1.0, 0.0), **want):
    return dict(name=name, img=img, px=np.asarray(px, float), level=level, T=np.asarray(T, float), d=tuple(float(v) for v in d),
                type=ftype, grad=tuple(grad), want=want)


def oracle_run(oracle, w, c, opts, d=None):
    f = oracle.cam2world(w.cam, c["px"][0], c["px"][1])
    fo = oracle.ref_feature(c["px"], f, c["level"], c["type"], c["grad"])
    d = c["d"] if d is None else d
    return oracle.find_epipolar_match(w.pr[c["img"]], w.pc[c["img"]], w.cam, fo, c["T"], d[0], d[1], d[2], opts)


def _bisect(pred, lo, hi, iters=80):
    """pred(lo) True, pred(hi) False -> (lo, hi) adjacent around the switch (geometric bisection)"""
    for _ in range(iters):
        mid = np.sqrt(lo * hi)
        if mid <= lo or mid >= hi:
            break
        lo, hi = (mid, hi) if pred(mid) else (lo, mid)
    return lo, hi


def _walk_case(oracle, w, probe, name, px, level, T, d_est, d_max, target):
    """d_min such that the oracle's n_steps == target exactly (n_steps falls as d_min rises towards d_max)"""
    c = _case(name, 0, px, level, T, (d_est, d_est, d_max))
    n_of = lambda dm: oracle_run(oracle, w, c, probe, (d_est, dm, d_max))[1].n_steps
    lo = d_est * 1e-5                                                  # near the epipole: n_steps >> any target
    _, up = _bisect(lambda dm: n_of(dm) >= target, lo, d_max)          # n_steps >= target below `up`
    lo2, _ = _bisect(lambda dm: n_of(dm) >= target + 1, lo, d_max)     # n_steps >= target + 1 up to lo2
    dm = np.sqrt(lo2 * up)
    return _case(name, 0, px, level, T, (d_est, dm, d_max), n_steps=target)


def _snap(px, level):
    return np.floor(np.asarray(px, float) / (1 << level)) * (1 << level)


def build_cases(oracle):
    """The case table (deterministic).  want: what the oracle must report for the case to test what it is named after."""
    w = world(oracle)
    probe = oracle.matcher_opts(NL, max_epi_search_steps=0)               # stops right after n_steps: cheap bisection
    z_of = lambda px: scenes.gt_depth(w.cfg, w.P0, px)[0]
    cases = []
    # exact walk lengths on every search level, far end at 1.5 x the depth and at infinity
    for level in range(NL):
        px = _snap((100, 200 + 8 * level), level)
        z = z_of(px)
        for d_max in (1.5 * z, INF_DEPTH):
            for t in WALK_TARGETS:
                cases.append(_walk_case(oracle, w, probe, "walk%d_L%d_%s" % (t, level, "inf" if d_max == INF_DEPTH else "fin"),
                                        px, level, T_SCENE, z, d_max, t))
                cases[-1]["want"]["search_level"] = level
        # epi_length just below and just above 2.0 (DIRECT / WALK switch)
        c = _case("epi2_L%d" % level, 0, px, level, T_SCENE, (z, z, 1.5 * z))
        el = lambda dm: oracle_run(oracle, w, c, probe, (z, dm, 1.5 * z))[1].epi_length
        above, below = _bisect(lambda dm: el(dm) >= 2.0, z * 1e-5, 1.5 * z)
        cases.append(_case("epi2_below_L%d" % level, 0, px, level, T_SCENE, (z, below, 1.5 * z), epi_below_2=True, search_level=level))
        cases.append(_case("epi2_above_L%d" % level, 0, px, level, T_SCENE, (z, above, 1.5 * z), epi_above_2=True, search_level=level))
    # the step limit and walks beyond 65,536 samples (level 0, starting inside the image, then leaving it); the 65,600-step
    # walk ends ~46,000 px away, beyond the +-32,767 px that a short2 pixel holds
    px = np.array([120.0, 240.0])
    for t in LONG_TARGETS:
        cases.append(_walk_case(oracle, w, probe, "long%d" % t, px, 0, T_SCENE, z_of(px), 1.5 * z_of(px), t))
    cases[-1]["want"]["beyond_short2"] = True
    # segments crossing the image border: leaving through the right, the bottom, starting outside and entering
    for name, p, T, lvl in (("border_right", (600, 240), T_SCENE, 0), ("border_right_L1", (596, 120), T_SCENE, 1),
                            ("border_bottom", (320, 460), T_Y, 0), ("border_top", (320, 10), [0, 0.1, 0.0005] + IDENT, 0)):
        p = _snap(p, lvl)
        z = z_of(p)
        cases.append(_case(name, 0, p, lvl, T, (z, 0.25 * z, 1.5 * z)))
    cases.append(_case("border_enter_left", 1, (6, 240), 0, T_X, (2.0, 26.25 / 30, 26.25 / 1)))
    # NaN depth ranges and a NaN estimate
    p = np.array([300.0, 200.0]); z = z_of(p)
    for name, d in (("nan_dmin", (z, np.nan, 1.5 * z)), ("nan_dmax", (z, 0.5 * z, np.nan)), ("nan_both", (z, np.nan, np.nan)),
                    ("nan_dest", (np.nan, 0.5 * z, 1.5 * z)), ("inf_dmax", (z, 0.5 * z, INF_DEPTH))):
        cases.append(_case(name, 0, p, 0, T_SCENE, d))
    # edgelets: gradients at several angles to the (near-horizontal) epipolar line, the filter's threshold cos = 0.7 between
    for k, ang in enumerate((0.0, 0.6, 0.79, 0.8, 1.2, np.pi / 2)):
        p = _snap((150 + 40 * k, 150), k % 3)
        z = z_of(p)
        cases.append(_case("edgelet%d" % k, 0, p, k % 3, T_SCENE, (z, 0.6 * z, 1.5 * z), ftype=1, grad=(np.cos(ang), np.sin(ang))))
    # ties: the current image repeats every PERIOD px along x and T_X moves along x, so the best score recurs every PERIOD px
    # of the walk (tie partners ~18.6 steps apart: other lanes of the group, both sides of sample 32 when the walk is long enough)
    fxt = w.cfg["fx"] * T_X[0]                                            # shift (px) = fx * tx / z
    for k, (s_lo, s_hi) in enumerate(((1, 40), (4, 44), (7, 50), (10, 90), (2, 30))):
        p = (200 + 17 * k, 120 + 40 * k)
        cases.append(_case("tie%d" % k, 1, p, 0, T_X, (2.0, fxt / s_hi, fxt / s_lo), tie=True))
    # flat reference patch against a flat image: every sample scores 0, the first non-repeated in-frame sample wins
    cases.append(_case("flat_inside", 2, (200, 200), 0, T_X, (2.0, fxt / 60, fxt / 3), flat=True))
    cases.append(_case("flat_enter", 2, (6, 200), 0, T_X, (2.0, fxt / 60, fxt / 1), flat=True))
    return cases


def tie_structure(oracle, c, e):
    """Scores of the (horizontal, one pixel per step or less) walk of a tie case from the image itself: the pixels that reach the
    minimum and the approximate step index of each.  Checks the replica against the oracle's n_evals and zmssd_best."""
    w = world(oracle)
    cam = w.cam
    f = oracle.cam2world(cam, c["px"][0], c["px"][1])
    d_est, d_min, d_max = c["d"]
    xs = [cam.fx * (f[0] * d + c["T"][0]) / (f[2] * d) + cam.cx for d in (d_max, d_min)]     # B (start), A (end)
    y = int(cam.fy * f[1] / f[2] + cam.cy + 0.5)
    step = (xs[1] - xs[0]) / e.n_steps
    img = w.cur_imgs[c["img"]].astype(np.int64)
    patch = np.array(e.patch[:], np.int64)
    a, aa = patch.sum(), (patch * patch).sum()
    scores = {}
    for x in range(int(xs[0] - step + 0.5), int(xs[1] - step + 0.5) + 1):     # samples B + (i - 1) step, i = 0 .. n_steps
        if not (8 <= x < cam.width - 8 and 8 <= y < cam.height - 8):
            continue
        b_ = img[y - 4:y + 4, x - 4:x + 4].ravel()
        b, bb, ab = b_.sum(), (b_ * b_).sum(), (b_ * patch).sum()
        scores[x] = int(aa - 2 * ab + bb - int((a * a - 2 * a * b + b * b) / 64))
    assert len(scores) == e.n_evals, (c["name"], len(scores), e.n_evals)
    best = min(scores.values())
    assert best == e.zmssd_best
    tied = sorted(x for x, s in scores.items() if s == best)
    steps = [int(np.ceil((x - 0.5 - xs[0]) / step)) + 1 for x in tied]   # first sample whose pixel is x (approximately)
    return tied, steps


def test_case_table_reaches_its_targets(oracle):
    """CPU: every edge the GPU tests rely on is really in the case table, judged by the oracle's own outputs."""
    w = world(oracle)
    cases = build_cases(oracle)
    assert len({c["name"] for c in cases}) == len(cases)
    big = oracle.matcher_opts(NL, max_epi_search_steps=INT_MAX)
    got_steps, levels_walked, below, above, many_evals, ties_across_32, ties_across_lanes = set(), set(), set(), set(), 0, 0, 0
    for c in cases:
        ok, e = oracle_run(oracle, w, c, big)
        want = c["want"]
        if "n_steps" in want:
            assert e.n_steps == want["n_steps"], (c["name"], e.n_steps)
            got_steps.add((e.n_steps, e.search_level))
        if "search_level" in want:
            assert e.search_level == want["search_level"], (c["name"], e.search_level)
            if e.n_steps >= 2:
                levels_walked.add(e.search_level)
        if want.get("epi_below_2"):
            assert e.epi_length < 2.0 and e.epi_length > 2.0 - 1e-9
            below.add(e.search_level)
        if want.get("epi_above_2"):
            assert e.epi_length >= 2.0 and e.epi_length < 2.0 + 1e-9 and e.n_steps == 2
            above.add(e.search_level)
        if want.get("beyond_short2"):
            assert e.n_steps > 65536 and e.n_evals > 0
            f = oracle.cam2world(w.cam, c["px"][0], c["px"][1])
            d = c["d"][1]
            assert abs(w.cam.fx * (f[0] * d + c["T"][0]) / (f[2] * d) + w.cam.cx) > 32767
        if want.get("tie"):
            tied, steps = tie_structure(oracle, c, e)
            assert len(tied) >= 2, c["name"]
            ties_across_32 += steps[0] <= 30 and steps[-1] >= 34
            ties_across_lanes += len({s % 8 for s in steps}) > 1
            # the first pixel of the walk with the best score wins
            assert int(e.px_cur[0] + 0.5) == tied[0] or ok
        if want.get("flat"):
            assert e.zmssd_best == 0 and e.n_evals > 1
        many_evals += e.n_evals > 64
    for level in range(NL):
        for t in WALK_TARGETS:
            assert (t, level) in got_steps, (t, level)
    for t in LONG_TARGETS:
        assert (t, 0) in got_steps, t
    assert levels_walked == below == above == set(range(NL))
    assert many_evals >= 3 and ties_across_32 >= 1 and ties_across_lanes >= 1


def _compare(g, ok, e, name):
    assert g["success"] == ok and g["reject"] == e.reject, (name, g["success"], ok)
    assert g["n_steps"] == e.n_steps, (name, g["n_steps"], e.n_steps)
    if e.reject:
        return
    assert g["search_level"] == e.search_level, name
    assert g["A_cur_ref"].tobytes() == np.array(e.A_cur_ref[:]).tobytes(), name
    assert g["epi_length"] == e.epi_length or (np.isnan(g["epi_length"]) and np.isnan(e.epi_length)), name
    assert np.array_equal(g["patch_with_border"], np.array(e.patch_with_border[:], np.uint8)), "%s: warped patch differs" % name
    assert np.array_equal(g["patch"], np.array(e.patch[:], np.uint8)), name
    assert g["zmssd_best"] == e.zmssd_best, (name, g["zmssd_best"], e.zmssd_best)
    assert g["n_evals"] == e.n_evals, (name, g["n_evals"], e.n_evals)
    if ok:
        assert np.abs(g["px_cur"] - np.array(e.px_cur[:])).max() <= PX_TOL, name
        assert g["px_cur"].tobytes() == np.array(e.px_cur[:]).tobytes(), "%s: px_cur not bit-exact" % name
        assert abs(g["depth"] - e.depth) <= 1e-12 * e.depth, name


def _sweep_items():
    """items of one sweep of the persistent search grid on this device"""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * SEARCH_CTAS * 16


@pytest.mark.gpu
@pytest.mark.parametrize("subpix", [1, 0])
@pytest.mark.parametrize("align_1d", [0, 1])
def test_epipolar_edges_match_oracle(ctx, oracle, subpix, align_1d):
    """Every case under every step limit and both edgelet-filter settings; the table is replicated past one sweep of the
    persistent grid, so every group handles several items and reserves LK job slots across them: replicas byte-identical."""
    w = world(oracle)
    cases = build_cases(oracle)
    cam_g = scenes.cam_of(w.cfg, capi.Camera)
    reps = _sweep_items() // len(cases) + 2
    rid, cid = upload(ctx, w.ref_imgs, NL), upload(ctx, w.cur_imgs, NL)
    try:
        n = len(cases)
        px = np.array([c["px"] for c in cases])
        f1 = _feature_refs(oracle, w.cam, rid, px, [c["level"] for c in cases], np.array([c["T"] for c in cases]),
                           [c["img"] for c in cases], [c["img"] for c in cases], [c["type"] for c in cases], [c["grad"] for c in cases])
        ftrs = np.tile(f1, reps)
        d = np.tile(np.array([c["d"] for c in cases]), (reps, 1))
        assert len(ftrs) > _sweep_items()
        n_walk_long = n_ok = 0
        mismatches = []
        for filt in (1, 0):
            for limit in LIMITS:
                kw = dict(align_1d=align_1d, subpix_refinement=subpix, max_epi_search_steps=limit, epi_search_edgelet_filtering=filt)
                got = ctx.epipolar_match(cid, cam_g, ftrs, d, ctx.matcher_opts(NL, **kw))
                rows = got.view(np.uint8).reshape(reps, -1)
                assert (rows == rows[0]).all(), "replicas differ (limit %d, filtering %d)" % (limit, filt)
                opts_o = oracle.matcher_opts(NL, **kw)
                for i, c in enumerate(cases):
                    ok, e = oracle_run(oracle, w, c, opts_o)
                    try:
                        _compare(got[i], ok, e, "%s limit=%d filt=%d" % (c["name"], limit, filt))
                    except AssertionError as err:          # collected, so that one failure does not hide the others
                        mismatches.append(str(err))
                    n_walk_long += e.n_steps > 1023 and e.n_evals > 0
                    n_ok += ok
        assert not mismatches, "%d case runs differ from the oracle:\n%s" % (len(mismatches), "\n".join(mismatches))
        assert n_walk_long > 0 and n_ok > 0
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


@pytest.mark.gpu
@pytest.mark.parametrize("limit", [1000, 1500, INT_MAX])
@pytest.mark.parametrize("subpix,align_1d", [(0, 0), (0, 1), (1, 1)])
def test_seeds_update_edges_match_oracle(ctx, oracle, subpix, align_1d, limit):
    """The depth filter's path (seeds_geom_kernel -> search -> LK -> seeds_finish_kernel, with EPI_FOUND_UV_ONLY ->
    world2cam_uv when subpix_refinement = 0) on seeds whose ranges give the table's walk lengths, infinite far ends
    (z_inv_max clamped) and NaN ranges, against oracle.update_seed_with_frame."""
    w = world(oracle)
    cases = [c for c in build_cases(oracle) if c["img"] == 0 and c["type"] == 0 and np.allclose(c["T"], T_SCENE)]
    cam_g = scenes.cam_of(w.cfg, capi.Camera)
    seeds = np.zeros(len(cases), capi.seed_dt)
    for i, c in enumerate(cases):
        # mu = 1 / d_estimate; z_inv_min = mu + sqrt(sigma2) = 1 / d_min, so z_inv_max = 2 mu - 1 / d_min (clamped to 1e-8:
        # a far end at infinity for the long walks)
        d_est, d_min, _ = c["d"]
        s = Seed(10.0, 10.0, 0.5 if np.isnan(d_est) else 1.0 / d_est, 1.0 / 0.3, 0.0)
        s.sigma2 = float(np.float32((1.0 / d_min - s.mu) ** 2))
        seeds[i] = (s.a, s.b, s.mu, s.z_range, s.sigma2)
    rid, cid = upload(ctx, w.ref_imgs, NL), upload(ctx, w.cur_imgs, NL)
    try:
        px = np.array([c["px"] for c in cases])
        levels = [c["level"] for c in cases]
        ftrs = _feature_refs(oracle, w.cam, rid, px, levels, np.zeros(7))
        T_ref_w = np.tile(w.P0, (len(cases), 1))
        T_cur_w = np.array([w.P1, w.P1, w.P1])
        kw = dict(align_1d=align_1d, subpix_refinement=subpix, max_epi_search_steps=limit)
        got_seeds, obs = ctx.seeds_update(cid, cam_g, ftrs, T_ref_w, T_cur_w, ctx.matcher_opts(NL, **kw), 100.0, seeds)
        opts_o = oracle.matcher_opts(NL, **kw)
        n_long = n_upd = 0
        for i, c in enumerate(cases):
            s = Seed(*[float(seeds[i][k]) for k in ("a", "b", "mu", "z_range", "sigma2")])
            fo = oracle.ref_feature(px[i], ftrs[i]["f"], levels[i])
            st, epi = oracle.update_seed_with_frame(w.pr[0], w.pc[0], w.cam, fo, w.P0, w.P1, opts_o, 100.0, s, want_epi=True)
            o = obs[i]
            assert o["status"] == st, "%s: status %d vs %d" % (c["name"], o["status"], st)
            if st >= 3:
                assert o["search_level"] == epi.search_level, c["name"]
                assert o["zmssd_best"] == epi.zmssd_best and o["n_evals"] == epi.n_evals, (c["name"], o["n_evals"], epi.n_evals)
                assert o["epi_length"] == epi.epi_length or (np.isnan(o["epi_length"]) and np.isnan(epi.epi_length)), c["name"]
                n_long += epi.n_steps > 65536 and epi.n_evals > 0
            if st >= 4:
                assert abs(o["z"] - epi.depth) <= 1e-12 * epi.depth, c["name"]
                assert np.abs(o["px_cur"] - np.array(epi.px_cur[:])).max() <= PX_TOL, c["name"]
                n_upd += 1
            for k in ("a", "b", "mu", "z_range", "sigma2"):
                e_, g_ = np.float32(getattr(s, k)), got_seeds[i][k]
                assert (np.isnan(e_) and np.isnan(g_)) or abs(g_ - e_) <= SEED_REL_TOL * abs(e_), (c["name"], k, g_, e_)
        assert n_upd > 0
        assert (n_long > 0) == (limit == INT_MAX)
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)


@pytest.mark.gpu
def test_negative_step_limit_rejected(ctx, oracle):
    """max_epi_search_steps is the reference's size_t: a negative value is an argument error, not "no limit"."""
    w = world(oracle)
    cam_g = scenes.cam_of(w.cfg, capi.Camera)
    rid, cid = upload(ctx, w.ref_imgs[:1], NL), upload(ctx, w.cur_imgs[:1], NL)
    try:
        c = build_cases(oracle)[0]
        ftrs = _feature_refs(oracle, w.cam, rid, c["px"][None], [c["level"]], c["T"])
        bad = ctx.matcher_opts(NL, max_epi_search_steps=-1)
        with pytest.raises(capi.Svob200Error, match="negative max_epi_search_steps"):
            ctx.epipolar_match(cid, cam_g, ftrs, np.array([c["d"]]), bad)
        with pytest.raises(capi.Svob200Error, match="negative max_epi_search_steps"):
            ctx.seeds_update(cid, cam_g, ftrs, w.P0[None], w.P1[None], bad, 100.0, np.zeros(1, capi.seed_dt))
        ao, h = capi.AlignOpts(3, 2, 30, 1e-6), C.c_void_p()
        rc = ctx.L.svob200_tracker_create(ctx.h, C.byref(cam_g), 1, NL, C.byref(ao), C.byref(bad), 100.0, 2.4, 0.3, 2, C.byref(h))
        assert rc == ERR_ARG and not h.value
        with pytest.raises(capi.Svob200Error, match="negative max_epi_search_steps"):
            ctx.epipolar_match(cid, cam_g, ftrs, np.array([c["d"]]), ctx.matcher_opts(NL, max_epi_search_steps=-(2 ** 31)))
    finally:
        ctx.frame_release(rid); ctx.frame_release(cid)
