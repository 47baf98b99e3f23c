#!/usr/bin/env python
"""bench.py — front-end frames/s of the B200-native SVO tracking front end (and the CPU reference arm).

Workload (BASELINE.json configs[4] built from configs[1]): a batch of independent synthetic
640x480 sequences (C2 shape: 4-level pyramid, 120 map features, 768 depth-filter seeds), sharded
over the GPUs of one node (strong scaling: the total number of sequences is fixed).  One step =
one frame of every sequence through pyramid -> sparse image alignment -> reprojection refinement ->
depth-filter seed update (svob200_tracker_step).  `value` times the steps with every input already
resident in HBM; `e2e` times the same steps through the C ABI with HOST (pinned) buffers, the H2D
copy of the frames + per-step inputs and the D2H read of the per-sequence results inside the timed
region.  The single-stream latency (one sequence, p50 / p95 per frame, C2 / C3 / C4 shapes) is reported in `latency`;
`next_rows` times the callers either side of the path (SURVEY 8f: YUV input stage, FAST, reprojector, pose and structure
optimisers, seed initialisation) on the device next to the reference's code on one host core.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--seqs TOTAL] [--dump-outputs DIR]
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the benchmark writes nothing into the tree it runs from (it may be read-only)

from android_svo_b200 import synth, frontend, sharding  # noqa: E402

METRIC = "front-end frames/s (pyramid + sparse align + refine + seed update), batched C2 sequences"
CFG_NAME = "C2"
TEX_SIZE = 2048
PPM = 400.0
PLANE_Z = 2.0
KF_RING, KF_MAX_N_KFS = 4, 3             # keyframes resident / DepthFilter::Options::max_n_kfs (--keyframe-every)
KF_INDEX = 0
POOL_INDICES = (36, 39, 42, 45)     # trajectory frames cycled (ping-pong) as the live stream
DEPTH_MEAN, DEPTH_MIN = 2.4, 1.2
DEPTH_MIN_YOUNG = 0.3                  # --seed-regime young: a wide depth prior (z_range = 1 / 0.3), so a fresh seed's epipolar segment is tens of pixels long
CHAIN_CELL, CHAIN_MAX_FTS = 30, 120   # Config::gridSize / maxFts defaults (config.cpp)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "dropin"],
                    help="b200: the CUDA path; reference: the reference's own CPU code; dropin: the reference's C++ harness linked over the "
                         "B200 drop-in (libsvo_dropin.so) next to the same harness over the reference's TUs, per-frame latency")
    ap.add_argument("--seed-regime", default="steady", choices=["steady", "young"],
                    help="steady: finished seeds are re-initialised (stationary workload, most seeds near convergence); young: EVERY seed is "
                         "re-initialised after every frame, so each update walks a long epipolar segment (north_star kernel 4)")
    ap.add_argument("--seqs", type=int, default=4096, help="total number of independent sequences (all GPUs)")
    ap.add_argument("--cpu-seqs", type=int, default=0, help="sequences in the CPU sample (0 = 4 per host thread)")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (ncu captures: only full-batch launches remain)")
    ap.add_argument("--chain", action="store_true", help="run the step in chain mode in BOTH arms: reprojector grid rules (cell 30, maxFts 120) + "
                    "pose optimiser between alignment and the depth filter (FrameHandlerMono::processFrame Steps 2-3)")
    ap.add_argument("--no-widen", action="store_true", help="skip the timing of the SURVEY 8f operators (reprojector, optimizers, YUV, seed init)")
    ap.add_argument("--keyframe-every", type=int, default=0, metavar="K",
                    help="insert a keyframe every K frames INSIDE the timed region, in both arms (svob200_tracker_add_keyframe / "
                         "DepthFilter::addKeyframe: occupancy, FAST + Shi-Tomasi + grid, seed initialisation; seeds of up to 4 keyframes, "
                         "ageing by max_n_kfs = 3, finished seeds leave the pool): FAST shows up in a step time")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (the per-sequence step records and a fixed, "
                         "seeded sample of the seed states; rank 0's sequences) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def ping_pong(n_pool, n_steps):
    """frame-pool indices visited so that consecutive frames are adjacent in time: 0,1,2,3,2,1,0,1,..."""
    order, i, d = [0], 0, 1
    while len(order) < n_steps + 1:
        if i + d < 0 or i + d >= n_pool:
            d = -d
        i += d
        order.append(i)
    return order


# ------------------------------------------------------------------ batched numpy geometry (setup only)
def poses_for(seq_ids, indices):
    """T_f_w[seq, frame] for the given trajectory frame indices."""
    n = max(indices) + 1
    return np.stack([synth.trajectory(n, seed=0x00C0FFEE + int(s))[list(indices)] for s in seq_ids])


def q_rot_many(q, p):
    """rotate points p[...,3] by quaternions q[...,4] (x,y,z,w)"""
    qv = q[..., :3]
    uv = np.cross(qv, p)
    uv = uv + uv
    return p + q[..., 3:4] * uv + np.cross(qv, uv)


def se3_inverse_many(T):
    qi = np.concatenate([-T[..., 3:6], T[..., 6:7]], -1)
    return np.concatenate([-q_rot_many(qi, T[..., :3]), qi], -1)


def backproject_many(cfg, T_f_w, px):
    """px[B,N,2] seen from T_f_w[B,7] -> world points on the plane z = PLANE_Z"""
    Tw = se3_inverse_many(T_f_w)
    d = np.stack([(px[..., 0] - cfg["cx"]) / cfg["fx"], (px[..., 1] - cfg["cy"]) / cfg["fy"], np.ones(px.shape[:-1])], -1)
    d = q_rot_many(Tw[:, None, 3:], d)
    s = (PLANE_Z - Tw[:, None, 2]) / d[..., 2]
    return Tw[:, None, :3] + s[..., None] * d


def project_many(cfg, T_f_w, pts):
    pc = q_rot_many(T_f_w[:, None, 3:], pts) + T_f_w[:, None, :3]
    return np.stack([cfg["fx"] * pc[..., 0] / pc[..., 2] + cfg["cx"], cfg["fy"] * pc[..., 1] / pc[..., 2] + cfg["cy"]], -1)


def natural_texture(size):
    """A texture with natural-image statistics for the detector: smooth shading (white noise, box-blurred to a ~24-px correlation
    length) plus a few dozen flat rectangles of random grey level (sharp edges and corners)."""
    rng = np.random.RandomState(12345)
    a = rng.randint(0, 256, (size, size)).astype(np.float64)
    for _ in range(3):
        for ax in (0, 1):
            c = np.cumsum(np.concatenate([a.take(range(-12, 0), axis=ax), a, a.take(range(0, 13), axis=ax)], axis=ax), axis=ax)
            a = (np.take(c, range(25, 25 + size), axis=ax) - np.take(c, range(0, size), axis=ax)) / 25.0
    a = (a - a.min()) / (a.max() - a.min()) * 160.0 + 40.0
    for _ in range(60):
        x0, y0 = rng.randint(0, size - 200, 2)
        ww, hh = rng.randint(40, 200, 2)
        a[y0:y0 + hh, x0:x0 + ww] = rng.randint(20, 236)
    return np.clip(a, 0, 255).astype(np.uint8)


def select_batch(cells, thr, n):
    px = np.zeros((len(cells), n, 2))
    lv = np.zeros((len(cells), n), np.int32)
    for b in range(len(cells)):
        good = cells[b][cells[b]["score"].astype(np.float64) > thr]
        if len(good) < n:      # texture-poor view: recycle the available corners so every sequence has the same load
            good = np.resize(good, n)
        good = good[:n]
        px[b] = np.stack([good["x"], good["y"]], 1)
        lv[b] = good["level"]
    return px, lv


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi polled every 20 ms in a child process; stop(t0, t1) keeps the samples whose timestamp falls inside the
    load window [t0, t1] (host wall clock: warm-up + timed steps)."""

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        if self.p is not None:
            atexit.register(self.p.kill)     # a run that fails inside the load window must not leave the poller behind

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, n_all = [], [], set(), 0
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f")
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            n_all += 1
            if t0 is not None and not (t0 <= ts <= t1):
                continue
            sm.append(clk); mx.append(cmax)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm), "samples_total": n_all}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------ CPU arm (reference / oracle port)
CPU_FRAMES_PER_STEP = 16   # a CPU "step" = this many consecutive frames of every sampled sequence (bounded sample, ~10-30 core-s per run)


def cpu_arm(cfg_name, n_seqs, steps, warmup, threads, inner=CPU_FRAMES_PER_STEP, chain=False, regime="steady", o3=False, dropin=False, kf_every=0,
            two_threads=False):
    """Times the front-end step of `n_seqs` independent sequences on the host cores.  Uses the real
    reference (oracle/_ref/libsvo_ref.so; o3: the -O3 / AVX2 / FMA build of the same sources; dropin: the same harness over
    the B200 drop-in) when it was built, else the C restatement.  One timed step = `inner` consecutive frames of every
    sequence, one worker task per sequence.  Every frame is timed on its own (perf_counter around the step call), and the
    reference harness splits it per operator with std::chrono::steady_clock (BASELINE.md section 3)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.pyoracle import Oracle, Ref, Cam, OracleSeq, RefSeq
    cfg = synth.CONFIGS[cfg_name]
    oracle, ref = Oracle(), Ref(o3=o3, dropin=dropin)
    kind = "reference" if ref.available() else "port"
    if dropin:
        if not ref.available():
            raise RuntimeError("oracle/_ref/libsvo_dropin.so is missing")
        kind = "dropin"
    cam = Cam.make(cfg["w"], cfg["h"], cfg["fx"], cfg["fy"], cfg["cx"], cfg["cy"])
    tex = synth.make_texture(TEX_SIZE)
    idx = (KF_INDEX,) + POOL_INDICES
    poses = poses_for(range(4096, 4096 + n_seqs) if n_seqs == 1 else range(n_seqs), idx)
    fc, ft, sc, st = frontend.DETECT[cfg_name]
    reseed = 2 if regime == "young" else 1

    def setup(i):
        imgs = [oracle.synth_render(tex, PPM, PLANE_Z, cam, poses[i, k]) for k in range(len(idx))]
        pyr = oracle.pyramid(imgs[0], cfg["n_levels"])
        _, fcells = oracle.fast_detect(pyr, cfg["n_pyr"], fc, ft)
        _, scells = oracle.fast_detect(pyr, cfg["n_pyr"], sc, st)
        kf = frontend.keyframe_setup(cfg, poses[i, 0], fcells, scells, ft, st, PLANE_Z, recycle=True)
        args = (cam, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"], 100.0, DEPTH_MEAN,
                DEPTH_MIN_YOUNG if regime == "young" else DEPTH_MIN, reseed)
        if kf_every:
            args = args[:-1] + (3,)          # the reference's list semantics: finished seeds leave the list
        s = RefSeq(ref, *args) if kind != "port" else OracleSeq(oracle, *args)
        if two_threads:
            s.set_threaded()             # the reference's native layout: the depth filter in its own thread (reference builds only)
        if kf_every:
            if kind != "port":
                s.set_pool(KF_RING, KF_MAX_N_KFS, 3, sc, cfg["n_pyr"], st)
            else:
                s.set_pool(KF_RING, KF_MAX_N_KFS, 3); s.set_detector(sc, cfg["n_pyr"], st)
        s.set_keyframe(imgs[0], poses[i, 0], kf["kf_px"], kf["kf_level"], kf["pt_world"], kf["seed_px"], kf["seed_level"])
        if chain:
            s.set_chain(CHAIN_CELL, CHAIN_MAX_FTS, 1)
        s.set_last(imgs[1])
        last_px = [frontend.project_many(cfg, poses[i, 1 + k], kf["pt_world"]) for k in range(len(POOL_INDICES))]
        return s, imgs[1:], last_px

    frame_s = [[] for _ in range(n_seqs)]
    with ThreadPoolExecutor(threads) as ex:
        seqs = list(ex.map(setup, range(n_seqs)))
        order = ping_pong(len(POOL_INDICES), (warmup + steps) * inner)

        def run_seq(i, k):
            st = None
            for j in range(k * inner, (k + 1) * inner):
                a, b = order[j], order[j + 1]
                t0 = time.perf_counter()
                st = seqs[i][0].step(seqs[i][1][b], poses[i, 1 + a], seqs[i][2][a])
                if kf_every and (j + 1) % kf_every == 0:
                    seqs[i][0].add_keyframe(DEPTH_MEAN, DEPTH_MIN)
                frame_s[i].append(time.perf_counter() - t0)
            return st

        def step_all(k):
            return list(ex.map(lambda i: run_seq(i, k), range(n_seqs)))

        for k in range(warmup):
            step_all(k)
        for f in frame_s:
            del f[:]
        if kind != "port":
            for s, _, _ in seqs:
                s.timing()
        t0 = time.perf_counter()
        for k in range(warmup, warmup + steps):
            stats = step_all(k)
        if two_threads:
            for s, _, _ in seqs:
                s.drain()                # the timed region ends when the depth-filter thread has consumed every frame
        dt = time.perf_counter() - t0
    tracked = float(np.mean([s.n_tracked for s in stats]))
    ops = None
    if kind != "port":
        acc = {}
        for s, _, _ in seqs:
            for k, v in s.timing().items():
                acc[k] = acc.get(k, 0.0) + v
        n = max(acc.pop("steps"), 1)
        ops = {k + "_ms": round(v / n * 1e3, 4) for k, v in acc.items()}
    for s, _, _ in seqs:
        s.close()
    ms = np.concatenate([np.array(f) for f in frame_s]) * 1e3
    return dict(kind=kind, fps=n_seqs * steps * inner / dt, seconds=dt, n_seqs=n_seqs, tracked=tracked, inner=inner,
                p50_ms=float(np.median(ms)), p95_ms=float(np.percentile(ms, 95)), mean_ms=float(ms.mean()), frames=int(len(ms)), per_operator=ops)


def cpu_two_threads(cfg_name, regime="steady", frames=96):
    """The reference's native layout on TWO host threads: tracking (pyramid, alignment, refinement) in one, DepthFilter::updateSeedsLoop in
    the other (depth_filter.cpp:63-67); the tracking thread is paced so that the filter's queue never drops a frame."""
    r = cpu_arm(cfg_name, 1, frames // 16, 1, 1, regime=regime, two_threads=True)
    return {"frames_per_s": round(r["fps"], 1), "ms_per_frame": round(1e3 / r["fps"], 4), "tracking_thread_p50_ms": round(r["p50_ms"], 4),
            "tracking_thread_p95_ms": round(r["p95_ms"], 4), "kind": r["kind"], "cores": 2,
            "sample": "1 sequence x %d frames (+16 warm-up), tracking thread + depth-filter thread, no dropped frames; throughput over the whole run "
                      "incl. draining the filter's queue; the tracking-thread latency includes waiting for a queue slot" % r["frames"]}


def cpu_latency(cfg_name, chain=False, regime="steady", o3=False, frames=48):
    """The reference's native single-stream mode: ONE sequence on ONE host thread, every frame timed; p50 / p95 over `frames`
    frames after 16 warm-up frames, with the harness's steady_clock split per operator."""
    r = cpu_arm(cfg_name, 1, frames // 16, 1, 1, chain=chain, regime=regime, o3=o3)
    out = {"p50_ms": round(r["p50_ms"], 4), "p95_ms": round(r["p95_ms"], 4), "mean_ms": round(r["mean_ms"], 4), "kind": r["kind"], "cores": 1,
           "build": "-O3 -march=x86-64-v3 (AVX2 + FMA), contraction allowed" if o3 else "-O2, the reference's CMake flags (baseline x86-64, no FMA)",
           "sample": "1 sequence x %d frames timed one by one (+16 warm-up frames), 1 thread, depth filter synchronous" % r["frames"]}
    if r["per_operator"]:
        out["per_operator_mean"] = r["per_operator"]
    return out


# ------------------------------------------------------------------ GPU arm
def pinned_array(ctx, shape, dtype):
    import ctypes as C
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    ctx._ck(ctx.L.svob200_host_alloc_pinned(ctx.h, n, C.byref(p)))
    buf = (C.c_char * n).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p.value


class GpuWorkload:
    """Everything the timed loops need, resident: tracker, frame pool on device + pinned host, per-step inputs."""

    def __init__(self, ctx, capi, cfg, seq_ids, tex_dev=None, cfg_name=CFG_NAME, chain=False, regime="steady", kf_every=0):
        self.ctx, self.capi, self.cfg = ctx, capi, cfg
        B = len(seq_ids)
        self.B = B
        w, h, N, S = cfg["w"], cfg["h"], cfg["n_features"], cfg["n_seeds"]
        cam = capi.Camera.make(w, h, cfg["fx"], cfg["fy"], cfg["cx"], cfg["cy"])
        self.cam = cam
        idx = (KF_INDEX,) + POOL_INDICES
        poses = poses_for(seq_ids, idx)                         # [B, 1+F, 7]
        self.poses = poses
        own_tex = tex_dev is None
        if own_tex:
            tex = synth.make_texture(TEX_SIZE)
            tex_dev = ctx.dev_alloc(tex.nbytes)
            ctx.dev_upload(tex_dev, tex)
        self.tex_dev, self.own_tex = tex_dev, own_tex
        F = len(POOL_INDICES)
        img_bytes = w * h
        # frame pool on the device (dense, stride = w) and in pinned host memory
        self.pool_dev = [ctx.dev_alloc(B * img_bytes) for _ in range(F)]
        self.pool_host = []
        for k in range(F):
            ctx.synth_render(tex_dev, TEX_SIZE, PPM, PLANE_Z, cam, poses[:, 1 + k], self.pool_dev[k])
            arr, ptr = pinned_array(ctx, (B, h, w), np.uint8)
            ctx.dev_download(arr, self.pool_dev[k])
            self.pool_host.append((arr, ptr))
        # keyframes: render, detect (GPU FAST), select features / seeds
        kf_dev = ctx.dev_alloc(B * img_bytes)
        ctx.synth_render(tex_dev, TEX_SIZE, PPM, PLANE_Z, cam, poses[:, 0], kf_dev)
        self.kf_host = np.zeros((B, h, w), np.uint8)
        ctx.dev_download(self.kf_host, kf_dev)
        ctx.dev_free(kf_dev)
        fid = 7
        ctx.frame_create(fid, B, w, h, cfg["n_levels"])
        ctx.frame_upload(fid, self.kf_host)
        fc, ft, sc, st = frontend.DETECT[cfg_name]
        fcells, _ = ctx.fast_detect(fid, cfg["n_pyr"], fc, ft)
        scells, _ = ctx.fast_detect(fid, cfg["n_pyr"], sc, st)
        ctx.frame_release(fid)
        kf_px, kf_level = select_batch(fcells, ft, N)
        seed_px, seed_level = select_batch(scells, st, S)
        pt_world = backproject_many(cfg, poses[:, 0], kf_px)
        self.kf = dict(kf_px=kf_px, kf_level=kf_level, pt_world=pt_world, seed_px=seed_px, seed_level=seed_level)
        self.trk = capi.Tracker(ctx, cam, B, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"], 100.0,
                                DEPTH_MEAN, DEPTH_MIN_YOUNG if regime == "young" else DEPTH_MIN, 2 if regime == "young" else 1)
        self.kf_every = kf_every
        self.kf_ms = []
        if kf_every:
            n_cells = -(-w // sc) * -(-h // sc)
            self.trk.set_seed_pool(S + (KF_RING - 1) * n_cells, KF_RING, KF_MAX_N_KFS, 3)
            self.trk.set_detector(sc, cfg["n_pyr"], st)
        self.trk.set_keyframe(self.kf_host, poses[:, 0], np.arange(B + 1) * N, kf_px.reshape(-1, 2), kf_level.reshape(-1),
                              pt_world.reshape(-1, 3), np.arange(B + 1) * S, seed_px.reshape(-1, 2), seed_level.reshape(-1))
        if chain:
            self.trk.set_chain(CHAIN_CELL, CHAIN_MAX_FTS, 1)
        # per-step inputs for every pool frame used as "last": pose + pixel of every map point
        self.in_host, self.in_dev = [], []
        for k in range(F):
            T = np.ascontiguousarray(poses[:, 1 + k])
            lp = np.ascontiguousarray(project_many(cfg, T, pt_world).reshape(-1, 2))
            hT, pT = pinned_array(ctx, T.shape, np.float64); hT[...] = T
            hp, pp = pinned_array(ctx, lp.shape, np.float64); hp[...] = lp
            dT, dp = ctx.dev_alloc(T.nbytes), ctx.dev_alloc(lp.nbytes)
            ctx.dev_upload(dT, T); ctx.dev_upload(dp, lp)
            self.in_host.append((pT, pp)); self.in_dev.append((dT, dp))
        self.stats_host, self.stats_ptr = pinned_array(ctx, (B,), capi.step_stats_dt)
        self.stats_dev = ctx.dev_alloc(self.stats_host.nbytes)
        self.h2d_bytes = B * img_bytes + B * 56 + B * N * 16
        self.d2h_bytes = self.stats_host.nbytes
        self.reset()

    def reset(self):
        self.trk.set_last(self.pool_dev[0], mem=self.capi.MEM_DEVICE, stride=self.cfg["w"])
        self.pos = 0

    def close(self):
        """release the tracker and every device / pinned buffer of this workload"""
        if self.trk is None:
            return
        self.ctx.sync()
        self.trk.close()
        self.trk = None
        for d in self.pool_dev + [x for pair in self.in_dev for x in pair] + [self.stats_dev]:
            self.ctx.dev_free(d)
        if self.own_tex:
            self.ctx.dev_free(self.tex_dev)
        for _, ptr in self.pool_host:
            self.ctx._ck(self.ctx.L.svob200_host_free_pinned(self.ctx.h, ptr))
        for pair in self.in_host:
            for ptr in pair:
                self.ctx._ck(self.ctx.L.svob200_host_free_pinned(self.ctx.h, ptr))
        self.ctx._ck(self.ctx.L.svob200_host_free_pinned(self.ctx.h, self.stats_ptr))
        self.pool_dev, self.pool_host, self.in_dev, self.in_host = [], [], [], []

    def step(self, order, k, mem):
        a, b = order[k], order[k + 1]
        w = self.cfg["w"]
        if mem == self.capi.MEM_DEVICE:
            self.trk.step_raw(self.pool_dev[b], w, self.in_dev[a][0], self.in_dev[a][1], self.stats_dev, mem)
        else:
            self.trk.step_raw(self.pool_host[b][1], w, self.in_host[a][0], self.in_host[a][1], self.stats_ptr, mem)
        if self.kf_every and (k + 1) % self.kf_every == 0:
            t0 = time.perf_counter()
            self.kf_new, self.kf_dropped = self.trk.add_keyframe(DEPTH_MEAN, DEPTH_MIN)     # synchronises (the counts go back to the host)
            self.kf_ms.append((time.perf_counter() - t0) * 1e3)


def seed_workload_of(obs, capi, regime):
    """What the depth filter did in the last step (svob200_seed_obs of every seed): the epipolar-search load."""
    ev = obs["n_evals"]
    searched = obs["status"] >= capi.SEED_NO_MATCH
    direct = searched & (obs["epi_length"] < 2.0)
    walk = searched & (obs["epi_length"] >= 2.0)
    n = max(len(obs), 1)
    return {"regime": regime, "n_evals_mean": round(float(ev.mean()), 2), "n_evals_p50": float(np.percentile(ev, 50)), "n_evals_p95": float(np.percentile(ev, 95)),
            "n_evals_mean_walk": round(float(ev[walk].mean()), 2) if walk.any() else 0.0,
            "frac_direct": round(float(direct.sum()) / n, 4), "frac_walk": round(float(walk.sum()) / n, 4),
            "frac_not_searched": round(float((~searched).sum()) / n, 4),
            "frac_updated": round(float((obs["status"] >= capi.SEED_UPDATED).sum()) / n, 4),
            "note": "direct = epipolar segment shorter than 2 px (align2D at the midpoint, matcher.cpp:257-278); walk = ZMSSD over the segment"}


DUMP_MAX_SEEDS = 1 << 20      # 20 MB of float32 seed states: the dump stays well under 64 MB at any batch size


def dump_outputs(out_dir, stats, seeds):
    """The last timed step's results as float64 / float32 .npy files: every field of the step records of every sequence, and
    the seed states (a, b, mu, z_range, sigma2) of all pool slots, or of a fixed seeded sample of DUMP_MAX_SEEDS slots."""
    os.makedirs(out_dir, exist_ok=True)
    for name in stats.dtype.names:
        np.save(os.path.join(out_dir, "step_%s.npy" % name), stats[name].astype(np.float64))
    idx = np.arange(len(seeds))
    if len(idx) > DUMP_MAX_SEEDS:
        idx = np.sort(np.random.RandomState(0).choice(len(seeds), DUMP_MAX_SEEDS, replace=False))
    np.save(os.path.join(out_dir, "seeds.npy"), np.stack([seeds[k][idx] for k in seeds.dtype.names], 1).astype(np.float32))


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from android_svo_b200 import capi
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = capi.Context(local_rank)
    cfg = synth.CONFIGS[CFG_NAME]
    total, per, rng = sharding.shard(args.seqs, rank, world)     # contiguous block partition (SURVEY §8e)
    seq_ids = list(rng)
    t_setup = time.time()
    wl = GpuWorkload(ctx, capi, cfg, seq_ids, chain=args.chain, regime=args.seed_regime, kf_every=args.keyframe_every)
    t_setup = time.time() - t_setup
    K, W = args.steps, args.warmup
    order = ping_pong(len(POOL_INDICES), 2 * (W + K) + 8)

    def barrier():
        ctx.sync()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        return sharding.max_over_ranks(x, world, "cuda")

    # ---------------- value: inputs resident in HBM, CUDA events on the launching stream
    import datetime
    wl.reset()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        time.sleep(1.0)                     # nvidia-smi needs most of a second before its first sample
    t_load0 = datetime.datetime.now()
    for k in range(W):
        wl.step(order, k, capi.MEM_DEVICE)
    barrier()
    launches0 = ctx.launch_count()
    ctx.timer_start()
    for k in range(W, W + K):
        wl.step(order, k, capi.MEM_DEVICE)
    ms = ctx.timer_stop_ms()
    barrier()
    t_load1 = datetime.datetime.now()
    clocks = sampler.stop(t_load0, t_load1) if sampler else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed steps, %.0f ms" % ((t_load1 - t_load0).total_seconds() * 1e3)
    launches = ctx.launch_count() - launches0
    ms = max_over_ranks(ms)
    value = total * K / (ms * 1e-3)
    stats_dev_copy = np.zeros(wl.B, capi.step_stats_dt)
    ctx.dev_download(stats_dev_copy, wl.stats_dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats_dev_copy, wl.trk.seeds())

    # ---------------- stage breakdown (separate, untimed-for-the-headline pass)
    wl.trk.enable_profiling(True)
    stage_acc, n_prof = {}, 3
    for k in range(W + K, W + K + n_prof):
        wl.step(order, k, capi.MEM_DEVICE)
        for name, v in wl.trk.stage_ms().items():
            stage_acc[name] = stage_acc.get(name, 0.0) + v / n_prof
    obs = wl.trk.seed_obs()
    wl.trk.enable_profiling(False)
    mean_evals = float(obs["n_evals"].mean())
    seed_workload = seed_workload_of(obs, capi, args.seed_regime)
    N, S = cfg["n_features"], cfg["n_seeds"]
    iters_mean = float(stats_dev_copy["align_iters"].mean())
    # algorithmic bytes per launch (DESIGN.md §kernels; SURVEY.md §8d per-unit figures x units per launch)
    alg = {
        "frame+pyramid": wl.B * 408000.0,
        "sparse_align": wl.B * N * (857.0 * iters_mean + 36.0 * (cfg["max_level"] - cfg["min_level"] + 1)),
        "match_prepare": wl.B * N * 400.0,                       # 100 bilinear taps of the reference patch
        "match_refine": wl.B * N * (128.0 + 2 * 81.0),          # job record + ~2 LK iterations over a 9x9 window
        "seeds_search": wl.B * S * (400.0 + 64.0 * mean_evals),  # patch warp + ZMSSD windows along the epipolar segment
        "seeds_refine": wl.B * S * (128.0 + 2 * 81.0),
    }
    kernel_of = {"frame+pyramid": "pyramid_fused_kernel", "sparse_align": "sparse_align_kernel", "match_prepare": "match_prepare_kernel",
                 "match_refine": "lk_refine_kernel", "seeds_search": "epi_search_kernel", "seeds_refine": "lk_refine_kernel"}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    stages = {}
    for name, v in stage_acc.items():
        e = {"ms": round(v, 4)}
        if name in alg and v > 0:
            e["alg_GBps"] = round(alg[name] / (v * 1e-3) / 1e9, 2)
            e["hbm_frac"] = round(e["alg_GBps"] / peak, 4)
        stages[name] = e
    dom = max(alg.keys(), key=lambda n: stage_acc.get(n, 0.0))
    # dram bytes per launch from the committed `ncu --set full` capture (profiles/traffic.json: bytes per sequence)
    tj = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass

    def traffic_of(name):
        t = tj.get(kernel_of[name], {}).get("dram_bytes_per_sequence")
        return None if t is None else round(t * wl.B)

    def roof(name):
        a = alg[name] / (stage_acc[name] * 1e-3) / 1e9
        r = {"kernel": kernel_of[name], "bound": "hbm", "achieved": round(a, 2), "peak": peak, "unit": "GB/s", "frac": round(a / peak, 5),
             "traffic": traffic_of(name), "algorithmic_bytes": round(alg[name]), "peak_source": peak_src,
             "ms_per_launch": round(stage_acc[name], 4), "share_of_step": round(stage_acc[name] / max(sum(stage_acc.values()), 1e-9), 3)}
        ncu = tj.get(kernel_of[name], {}).get("ncu")
        if ncu:   # what actually bounds the kernel, from the committed `ncu --set full` capture (profiles/)
            r["ncu"] = {k: (round(v, 2) if isinstance(v, float) else v) for k, v in ncu.items()}
            r["ncu"]["source"] = tj[kernel_of[name]].get("source")
        return r

    roofline = roof(dom)
    roofline["note"] = ("dominant kernel of the step; it is integer-issue/L2-bound (ZMSSD dot products and LK on L2-resident windows), "
                        "so its HBM fraction is small by construction; the HBM-streaming kernel of the path is the pyramid: "
                        "see roofline_pyramid") if dom != "frame+pyramid" else "HBM-streaming kernel"
    roofline_pyr = roof("frame+pyramid")
    for name in stages:
        if name in alg:
            stages[name]["traffic"] = traffic_of(name)

    # ---------------- plain pinned H2D rate of this box (context for the PCIe-bound e2e number)
    t0 = time.perf_counter()
    for _ in range(3):
        ctx.dev_upload(wl.pool_dev[0], wl.pool_host[1][0])
    pcie = 3 * wl.pool_host[1][0].nbytes / (time.perf_counter() - t0) / 1e9
    ctx.dev_upload(wl.pool_dev[0], wl.pool_host[0][0])

    # ---------------- e2e: host (pinned) buffers through the C ABI, copies inside the timed region
    wl.reset()
    if args.no_e2e:
        for k in range(2):
            wl.step(order, k, capi.MEM_DEVICE)
        ctx.sync()
        ctx.dev_download(wl.stats_host, wl.stats_dev)
        e2e_s, order_last = float("nan"), order[2]
    else:
        for k in range(W):
            wl.step(order, k, capi.MEM_HOST)
        barrier()
        t0 = time.perf_counter()
        for k in range(W, W + K):
            wl.step(order, k, capi.MEM_HOST)
        ctx.sync()
        e2e_s = time.perf_counter() - t0
        barrier()
        e2e_s = max_over_ranks(e2e_s)
        order_last = order[W + K]
    e2e_value = total * K / e2e_s
    stats_last = wl.stats_host.copy()

    # ---------------- per-sequence statistics: NCCL gather over NVLink (SURVEY §8e), 64 B per sequence
    gt = wl.poses[:, 1 + order_last]
    perr = np.array([synth.pose_error(stats_last["T_cur_w"][b], gt[b]) for b in range(wl.B)])
    rec = sharding.gather_records(sharding.make_records(seq_ids, stats_last, perr), world, "cuda")
    seq_stats = sharding.summarize(rec)
    seq_stats["record_bytes"] = sharding.RECORD_BYTES

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8 pixels / f32 photometric / f64 geometry", "data": "synthetic",
            "config": {"workload": "C5: %d independent C2 sequences (640x480, 4-level pyramid, %d map features, %d seeds each), "
                                   "block-sharded over %d GPU(s); step = 1 frame of every sequence" % (total, N, S, world),
                       "sequences_total": total, "sequences_per_gpu": per, "frame_pool": list(POOL_INDICES),
                       "seed_regime": args.seed_regime,
                       "keyframe_every": args.keyframe_every or None,
                       "step": ("chain: reprojector grid rules (cell %d, maxFts %d) + pose optimiser between alignment and the depth filter"
                                % (CHAIN_CELL, CHAIN_MAX_FTS)) if args.chain else "refine every map point of the keyframe (batched superset of the reprojector)",
                       "l2": "inputs larger than L2 (%.0f MB of frames per step per GPU)" % (per * cfg["w"] * cfg["h"] / 1e6)},
            "e2e": {"skipped": "--no-e2e"} if args.no_e2e else {"value": round(e2e_value, 1), "unit": "frames/s", "h2d_bytes_per_step": int(wl.h2d_bytes * world),
                    "d2h_bytes_per_step": int(wl.d2h_bytes * world), "ms_per_step": round(e2e_s / K * 1e3, 4),
                    "h2d_GBps_per_gpu": round(wl.h2d_bytes / (e2e_s / K) / 1e9, 2), "pcie_h2d_GBps_measured": round(pcie, 2),
                    "note": "host-buffer path is PCIe-bound: the frame upload (307,200 B/frame) is chunked and overlapped with compute"},
            "gpu_launches": int(launches), "launches_per_step": int(launches // max(K, 1)),
            "clocks": clocks, "roofline": roofline, "roofline_pyramid": roofline_pyr, "stages": stages, "seed_workload": seed_workload,
            "zmssd_evals_per_s": round(float(obs["n_evals"].sum()) / max(stage_acc.get("seeds_search", 0.0), 1e-9) * 1e3, 1),
            "sequence_stats": seq_stats,
            "keyframes": None if not args.keyframe_every else {
                "every": args.keyframe_every, "ring": KF_RING, "max_n_kfs": KF_MAX_N_KFS,
                "add_keyframe_ms_host_wall_median": round(float(np.median(wl.kf_ms)), 3) if wl.kf_ms else None,
                "note": "wall time of svob200_tracker_add_keyframe incl. the join of the in-flight depth filter of the preceding step, the level-0 copy, "
                        "occupancy, FAST + Shi-Tomasi + grid over %d frames, seed initialisation and the read-back of the counts" % per,
                "new_seeds_mean": float(np.mean(wl.kf_new)) if wl.kf_ms else None, "dropped_mean": float(np.mean(wl.kf_dropped)) if wl.kf_ms else None},
            "setup_s": round(t_setup, 1),
        }
    return out, ctx, wl


def widen_rows(ctx, capi, wl, cfg, peak, steps=5, warm=2):
    """The callers either side of the hot path (SURVEY §8f), timed on the device over the same batch of sequences
    (CUDA events on the context's stream, inputs resident) next to the reference's own CPU code on one host core:
      yuv_pyramid      svob200_frame_upload_yuv420    YUV_420_888 -> gray -> pyramid, one fused kernel (HBM-bound)
      reproject_map    svob200_reproject_map          grid + batched findMatchDirect + per-cell / maxFts rules
      pose_optimize    svob200_pose_optimize          motion-only Gauss-Newton per frame
      points_optimize  svob200_points_optimize        Point::optimize for every map point (3 observations each)
      seeds_initialize svob200_seeds_initialize       occupancy + FAST + Shi-Tomasi + grid + Seed ctor"""
    import ctypes as C
    B, N, w, h = wl.B, cfg["n_features"], cfg["w"], cfg["h"]
    out = {}

    def timed(fn):
        for _ in range(warm):
            fn()
        ctx.sync()
        ctx.timer_start()
        for _ in range(steps):
            fn()
        return ctx.timer_stop_ms() / steps

    def dev(a):
        a = np.ascontiguousarray(a)
        d = ctx.dev_alloc(max(a.nbytes, 1))
        ctx.dev_upload(d, a)
        return d

    L, P, V = ctx.L, capi._ptr, C.c_void_p
    frees = []
    try:
        # ---- frames: keyframe batch (id 901) and a current batch (id 902) with the pose of pool frame 1
        ctx.frame_create(901, B, w, h, cfg["n_levels"]); ctx.frame_upload(901, wl.kf_host)
        ctx.frame_create(902, B, w, h, cfg["n_levels"])
        ctx._ck(L.svob200_frame_upload(ctx.h, 902, V(wl.pool_dev[1]), w, None, capi.MEM_DEVICE))
        T_cur = np.ascontiguousarray(wl.poses[:, 2]); T_kf = np.ascontiguousarray(wl.poses[:, 0])
        # ---- the pyramid kernel ALONE (device-memory bind of level 0 + one fused launch; in the step it shares the GPU with the
        #      previous frame's depth-filter stream, so its stage time there is not its own)
        lv = sum((w >> l) * (h >> l) for l in range(1, cfg["n_levels"]))
        alg_p = B * (w * h + lv)
        src = [wl.pool_dev[1], wl.pool_dev[2]]
        cnt = [0]

        def pyr_once():
            cnt[0] += 1
            ctx._ck(L.svob200_frame_bind(ctx.h, 902, V(src[cnt[0] & 1]), w, None))
        ms = timed(pyr_once)
        out["pyramid_alone"] = {"ms": round(ms, 4), "algorithmic_bytes": int(alg_p), "alg_GBps": round(alg_p / ms / 1e6, 1),
                                "hbm_frac": round(alg_p / ms / 1e6 / peak, 4), "bound": "hbm",
                                "note": "svob200_frame_bind (level 0 aliases the caller's device buffer, as in the tracker step), %d launches back to back, inputs alternate between two %d MB batches" % (steps, B * w * h >> 20)}
        ctx._ck(L.svob200_frame_upload(ctx.h, 902, V(wl.pool_dev[1]), w, None, capi.MEM_DEVICE))
        # ---- YUV input stage: Y = the live frame, neutral chroma (NV21 layout: one interleaved VU plane)
        d_y = wl.pool_dev[2]
        d_vu = ctx.dev_alloc(B * (h // 2) * w + 16); frees.append(d_vu)
        chroma = np.full(B * (h // 2) * w + 16, 128, np.uint8)
        ctx.dev_upload(d_vu, chroma)
        ctx.frame_create(903, B, w, h, cfg["n_levels"])
        ms = timed(lambda: ctx.frame_upload_yuv420(903, d_y, d_vu + 1, d_vu, w, w, 2, w * h, (h // 2) * w, mem=capi.MEM_DEVICE))
        lv = sum((w >> l) * (h >> l) for l in range(1, cfg["n_levels"]))
        alg = B * (w * h * 1.5 + w * h + lv)            # read Y + VU once, write gray once, write every coarser level once
        out["yuv_pyramid"] = {"ms": round(ms, 4), "frames_per_s": round(B / ms * 1e3, 1), "algorithmic_bytes": int(alg),
                              "alg_GBps": round(alg / ms / 1e6, 1), "hbm_frac": round(alg / ms / 1e6 / peak, 4), "bound": "hbm"}
        ctx.frame_release(903)
        # ---- reprojector: every map point of the keyframe, one observation each
        pts = np.zeros(B * N, capi.map_point_dt)
        pts["pos"] = wl.kf["pt_world"].reshape(-1, 3); pts["type"] = capi.POINT_UNKNOWN
        pts["obs_begin"] = np.arange(B * N); pts["obs_end"] = np.arange(B * N) + 1
        obs = np.zeros(B * N, capi.feature_ref_dt)
        obs["ref_frame_id"] = ctx.frame_slot(901); obs["ref_image"] = np.repeat(np.arange(B), N); obs["level"] = wl.kf["kf_level"].reshape(-1)
        px = wl.kf["kf_px"].reshape(-1, 2)
        obs["px"] = px
        fv = np.stack([(px[:, 0] - cfg["cx"]) / cfg["fx"], (px[:, 1] - cfg["cy"]) / cfg["fy"], np.ones(len(px))], 1)
        obs["f"] = fv / np.linalg.norm(fv, axis=1, keepdims=True); obs["grad"] = (1.0, 0.0)
        cell, max_fts = 30, 120
        n_cells = -(-w // cell) * -(-h // cell)
        d_T, d_off, d_pts, d_obs = dev(T_cur), dev(np.arange(B + 1, dtype=np.int32) * N), dev(pts), dev(obs)
        d_To = dev(np.repeat(T_kf, N, axis=0))
        d_res = ctx.dev_alloc(B * N * capi.reproj_result_dt.itemsize); d_win = ctx.dev_alloc(B * n_cells * 4); d_st = ctx.dev_alloc(B * 16)
        frees += [d_T, d_off, d_pts, d_obs, d_To, d_res, d_win, d_st]
        mo = ctx.matcher_opts(cfg["n_pyr"])
        ms = timed(lambda: ctx._ck(L.svob200_reproject_map(ctx.h, 902, C.byref(wl.cam), B, V(d_T), V(d_off), B * N, V(d_pts), B * N, V(d_obs), V(d_To),
                                                           cell, max_fts, C.byref(mo), V(d_res), V(d_win), V(d_st), capi.MEM_DEVICE)))
        st = np.zeros(B, capi.reproj_stats_dt); ctx.dev_download(st, d_st)
        res = np.zeros(B * N, capi.reproj_result_dt); ctx.dev_download(res, d_res)
        out["reproject_map"] = {"ms": round(ms, 4), "frames_per_s": round(B / ms * 1e3, 1), "points_per_frame": N,
                                "matches_mean": float(st["n_matches"].mean()), "trials_mean": float(st["n_trials"].mean())}
        # ---- pose optimizer on the matched features of every frame (alignment pose perturbed by the tracker's own error)
        ok = res["status"] == capi.REPROJ_MATCHED
        cnt = ok.reshape(B, N).sum(1)
        foff = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
        pxm = res["px"][ok]
        fm = np.stack([(pxm[:, 0] - cfg["cx"]) / cfg["fx"], (pxm[:, 1] - cfg["cy"]) / cfg["fy"], np.ones(len(pxm))], 1)
        fm /= np.linalg.norm(fm, axis=1, keepdims=True)
        d_foff, d_f, d_lv, d_pos = dev(foff), dev(fm), dev(res["search_level"][ok].astype(np.int32)), dev(pts["pos"][ok])
        d_Tp = ctx.dev_alloc(T_cur.nbytes); d_pr = ctx.dev_alloc(B * capi.pose_opt_result_dt.itemsize); d_out = ctx.dev_alloc(max(int(ok.sum()), 1))
        frees += [d_foff, d_f, d_lv, d_pos, d_Tp, d_pr, d_out]
        po = ctx.pose_opt_opts()

        def pose_run():
            ctx.dev_upload(d_Tp, T_cur)
            ctx._ck(L.svob200_pose_optimize(ctx.h, C.byref(wl.cam), B, V(d_foff), V(d_f), V(d_lv), V(d_pos), C.byref(po), V(d_Tp), V(d_pr), V(d_out), capi.MEM_DEVICE))
        ms = timed(pose_run)
        pr = np.zeros(B, capi.pose_opt_result_dt); ctx.dev_download(pr, d_pr)
        out["pose_optimize"] = {"ms": round(ms, 4), "frames_per_s": round(B / ms * 1e3, 1), "features_mean": float(cnt.mean()),
                                "iters_mean": float(pr["iters"].mean()), "error_final_px_median": float(np.median(pr["error_final"])),
                                "note": "includes the 229 KB pose re-upload per run"}
        # ---- structure optimisation: every map point seen from the keyframe and two live frames
        Tobs = np.stack([wl.poses[:, 0], wl.poses[:, 1], wl.poses[:, 3]], 1)              # [B, 3, 7]
        pw = wl.kf["pt_world"].reshape(B, N, 3)
        fb = np.zeros((B, N, 3, 3))
        for k in range(3):
            pc = q_rot_many(Tobs[:, None, k, 3:], pw) + Tobs[:, None, k, :3]
            fb[:, :, k] = pc / np.linalg.norm(pc, axis=-1, keepdims=True)
        d_ooff, d_To3, d_fb = dev(np.arange(B * N + 1, dtype=np.int32) * 3), dev(np.repeat(Tobs[:, None], N, axis=1).reshape(-1, 7)), dev(fb.reshape(-1, 3))
        pos0 = pw.reshape(-1, 3) + np.random.RandomState(1).normal(0, 0.01, (B * N, 3))
        d_p0 = ctx.dev_alloc(pos0.nbytes)
        frees += [d_ooff, d_To3, d_fb, d_p0]

        def pts_run():
            ctx.dev_upload(d_p0, pos0)
            ctx._ck(L.svob200_points_optimize(ctx.h, B * N, V(d_ooff), V(d_To3), V(d_fb), 20, 1e-10, V(d_p0), None, capi.MEM_DEVICE))
        ms = timed(pts_run)
        got = np.zeros_like(pos0); ctx.dev_download(got, d_p0)
        out["points_optimize"] = {"ms": round(ms, 4), "points_per_s": round(B * N / ms * 1e3, 1), "obs_per_point": 3,
                                  "median_error_m": float(np.median(np.linalg.norm(got - pw.reshape(-1, 3), axis=1))),
                                  "note": "includes the 11.8 MB start-position re-upload per run"}
        # ---- FAST + Shi-Tomasi + grid (SURVEY 8a a3/a4; keyframes only, so it is reported here and not in the step)
        fcell, fthr = frontend.DETECT[CFG_NAME][0], frontend.DETECT[CFG_NAME][1]
        fnc = -(-w // fcell) * -(-h // fcell)
        d_fc, d_fn = ctx.dev_alloc(B * fnc * 16), ctx.dev_alloc(B * 4)
        frees += [d_fc, d_fn]
        ms = timed(lambda: ctx._ck(L.svob200_fast_detect(ctx.h, 901, cfg["n_pyr"], fcell, fthr, None, V(d_fc), V(d_fn), capi.MEM_DEVICE)))
        alg = B * (408000.0 + fnc * 20)
        out["fast_detect"] = {"ms": round(ms, 4), "frames_per_s": round(B / ms * 1e3, 1), "Mpx_per_s": round(B * 408000 / ms / 1e3, 1),
                              "algorithmic_bytes": int(alg), "alg_GBps": round(alg / ms / 1e6, 1), "hbm_frac": round(alg / ms / 1e6 / peak, 4),
                              "bound": "integer ALU pipe (ncu r2b: ALU pipe 79 % busy, 2.4 M warp instructions per VGA frame; every pixel is scored with "
                                       "16-bit-lane VIMNMX3, 24 % of this texture's pixels are FAST corners)"}
        # ---- the same detector on a texture with natural-image statistics (smooth shading + a few objects with sharp edges: FAST's
        # share of corners is ~1 % there, against 24 % on the bench texture, whose blurred noise makes every fourth pixel a corner)
        nat = natural_texture(TEX_SIZE)
        d_nat = ctx.dev_alloc(nat.nbytes); frees.append(d_nat)
        ctx.dev_upload(d_nat, nat)
        d_nimg = ctx.dev_alloc(B * w * h); frees.append(d_nimg)
        ctx.synth_render(d_nat, TEX_SIZE, PPM, PLANE_Z, wl.cam, wl.poses[:, 0], d_nimg)
        ctx.frame_create(904, B, w, h, cfg["n_levels"])
        ctx._ck(L.svob200_frame_upload(ctx.h, 904, V(d_nimg), w, None, capi.MEM_DEVICE))
        ms_nat = timed(lambda: ctx._ck(L.svob200_fast_detect(ctx.h, 904, cfg["n_pyr"], fcell, fthr, None, V(d_fc), V(d_fn), capi.MEM_DEVICE)))
        fn = np.zeros(B, np.int32); ctx.dev_download(fn, d_fn)
        ctx.frame_release(904)
        out["fast_detect"]["natural_texture"] = {"ms": round(ms_nat, 4), "frames_per_s": round(B / ms_nat * 1e3, 1), "alg_GBps": round(alg / ms_nat / 1e6, 1),
                                                 "hbm_frac": round(alg / ms_nat / 1e6 / peak, 4), "features_mean": float(fn.mean())}
        # ---- seed initialisation on the keyframe batch
        d_eoff, d_epx = dev(np.arange(B + 1, dtype=np.int32) * N), dev(wl.kf["kf_px"].reshape(-1, 2))
        d_dm, d_dn = dev(np.full(B, DEPTH_MEAN, np.float32)), dev(np.full(B, DEPTH_MIN, np.float32))
        fc = frontend.DETECT[CFG_NAME][2]
        nc = -(-w // fc) * -(-h // fc)
        d_co, d_so, d_cn = ctx.dev_alloc(B * nc * 16), ctx.dev_alloc(B * nc * 20), ctx.dev_alloc(B * 4)
        frees += [d_eoff, d_epx, d_dm, d_dn, d_co, d_so, d_cn]
        ms = timed(lambda: ctx._ck(L.svob200_seeds_initialize(ctx.h, 901, cfg["n_pyr"], fc, frontend.DETECT[CFG_NAME][3], V(d_eoff), V(d_epx), V(d_dm), V(d_dn),
                                                              V(d_co), V(d_so), V(d_cn), capi.MEM_DEVICE)))
        cn = np.zeros(B, np.int32); ctx.dev_download(cn, d_cn)
        alg = B * (408000.0 + nc * 36)
        out["seeds_initialize"] = {"ms": round(ms, 4), "frames_per_s": round(B / ms * 1e3, 1), "new_seeds_mean": float(cn.mean()),
                                   "alg_GBps": round(alg / ms / 1e6, 1), "hbm_frac": round(alg / ms / 1e6 / peak, 4)}
    finally:
        for fid in (901, 902):
            try:
                ctx.frame_release(fid)
            except Exception:
                pass
        for d in frees:
            ctx.dev_free(d)
    return out


def widen_cpu(cfg):
    """The same operators in the reference's own code (oracle/_ref/libsvo_ref.so) on ONE host core, per frame / per
    point, on a bounded sample; the YUV stage is the oracle's port of the app's loop + cv2-equivalent gray (kind: port)."""
    from oracle.pyoracle import Oracle, Cam
    from oracle import pyoracle_map as pm
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import map_scenes as ms
    oracle = Oracle()
    om, rm = pm.OracleMap(oracle), pm.RefMap()
    out = {"cores": 1}
    w, h = cfg["w"], cfg["h"]
    fr = ms.yuv_frame(w, h, 1, 2, 0)
    t0 = time.perf_counter()
    for _ in range(5):
        g = om.yuv420_to_gray(fr["y"], fr["u"], fr["v"], fr["uv_stride"], 2, w, h, fr["y_stride"]); oracle.pyramid(g, cfg["n_levels"])
    out["yuv_pyramid_ms_per_frame"] = round((time.perf_counter() - t0) / 5 * 1e3, 3)
    if not rm.available():
        out["kind"] = "port (reference .so not built)"
        return out
    out["kind"] = "reference"
    full = dict(w=w, h=h, fx=cfg["fx"], fy=cfg["fy"], cx=cfg["cx"], cy=cfg["cy"], n_levels=cfg["n_levels"], n_pyr=cfg["n_pyr"])
    sc = ms.build_map_scene(oracle, cfg=full, seed=5, n_kf=1, cell=40, tex_size=1024, n_candidates=0, with_edgelets=False, bad_frac=0.0)
    cam = Cam.make(w, h, cfg["fx"], cfg["fy"], cfg["cx"], cfg["cy"])
    rm.config(cfg["n_pyr"], 30, 120)
    t0 = time.perf_counter()
    for _ in range(3):
        r = rm.reproject_map(sc["kf_imgs"], sc["T_kf"], sc["cur_img"], sc["T_cur"], cam, sc["points"], sc["obs"], 0)
    out["reproject_map_ms_per_frame"] = round((time.perf_counter() - t0) / 3 * 1e3, 3)
    out["reproject_map_points"] = int(len(sc["points"])); out["reproject_map_note"] = "includes building the Map and three Frame pyramids in the harness"
    s = ms.pose_opt_scene(cfg=full, seed=3, n=100)
    img = np.zeros((h, w), np.uint8)
    t0 = time.perf_counter()
    for _ in range(20):
        rm.pose_optimize(cam, img, s["px"], s["level"], s["pos"], s["T_init"])
    out["pose_optimize_ms_per_frame"] = round((time.perf_counter() - t0) / 20 * 1e3, 3)
    pts = ms.point_opt_scene(cfg=full, n_points=50, max_obs=3)
    t0 = time.perf_counter()
    for p in pts:
        rm.point_optimize(cam, img, p["T"], p["f"], p["pos0"])
    out["points_optimize_us_per_point"] = round((time.perf_counter() - t0) / len(pts) * 1e6, 1)
    out["points_optimize_note"] = "harness builds one Frame (pyramid) per observation: upper bound on the reference's cost"
    t0 = time.perf_counter()
    for _ in range(3):
        rm.initialize_seeds(cam, sc["kf_imgs"][0], cfg["n_pyr"], 20, 10.0, sc["obs"]["ftr"]["px_ref"], DEPTH_MEAN, DEPTH_MIN)
    out["seeds_initialize_ms_per_frame"] = round((time.perf_counter() - t0) / 3 * 1e3, 3)
    return out


LATENCY_DESC = {"C2": "C2: one 640x480 sequence, 4-level pyramid, 120 features, 768 seeds",
                "C3": "C3: one 752x480 sequence (EuRoC-shaped), 5-level pyramid, 300 features, 2,000 seeds",
                "C4": "C4: one 1920x1080 sequence (phone-shaped), 5-level pyramid, 1,000 features, 10,000 seeds"}


def latency_single(ctx, capi, name, n_frames=60, chain=False, regime="steady"):
    """Single-stream: one sequence, per-frame latency through the C ABI with host buffers (p50) and resident."""
    cfg = synth.CONFIGS[name]
    wl = GpuWorkload(ctx, capi, cfg, [4096], cfg_name=name, chain=chain, regime=regime)
    order = ping_pong(len(POOL_INDICES), n_frames + 30)
    res = {}
    for mode, mem in (("host_buffers", capi.MEM_HOST), ("resident", capi.MEM_DEVICE)):
        wl.reset()
        for k in range(10):
            wl.step(order, k, mem)
        ctx.sync()
        ts = []
        for k in range(10, 10 + n_frames):
            t0 = time.perf_counter()
            wl.step(order, k, mem)
            ctx.sync()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e3
        res[mode] = {"p50_ms": round(float(np.median(ts)), 4), "p95_ms": round(float(np.percentile(ts, 95)), 4),
                     "frames_per_s": round(1e3 / float(np.median(ts)), 1)}
    wl.trk.enable_profiling(True)
    acc = {}
    for k in range(5):
        wl.step(order, 10 + n_frames + k, capi.MEM_DEVICE)
        for n, v in wl.trk.stage_ms().items():
            acc[n] = acc.get(n, 0.0) + v / 5
    res["stages_ms_resident"] = {k: round(v, 4) for k, v in acc.items()}
    res["config"] = LATENCY_DESC[name]
    st = np.zeros(1, capi.step_stats_dt)
    ctx.dev_download(st, wl.stats_dev)
    res["tracked"] = int(st["n_tracked"][0]); res["matched"] = int(st["n_matched"][0]); res["seeds_updated"] = int(st["n_seeds_updated"][0])
    wl.close()
    return res


def dropin_line(args, cfg, threads):
    """--impl dropin: the reference's C++ harness (oracle/ref_harness.cpp: new Frame -> SparseImgAlign::run -> Matcher::findMatchDirect
    per map point -> DepthFilter::addFrame) linked over android_svo_b200/host/svo_b200_dropin.cpp, i.e. every operator call of the
    reference's own control flow lands in CUDA through the C ABI, timed per frame on ONE host thread next to the same harness over the
    reference's TUs.  Each drop-in call pays its own H2D / D2H and a synchronisation (INTEGRATION.md section 3): this is the number a
    maintainer gets by swapping the five TUs and changing nothing else."""
    frames = max(16, min(args.steps, 10) * 16)
    d = cpu_arm(CFG_NAME, 1, frames // 16, 1, 1, chain=args.chain, regime=args.seed_regime, dropin=True)
    r = cpu_arm(CFG_NAME, 1, frames // 16, 1, 1, chain=args.chain, regime=args.seed_regime)
    # the reference's native two-thread layout (tracking thread + DepthFilter::updateSeedsLoop thread) over both sets of TUs: the drop-in
    # serves the two threads from two svob200 contexts (two streams), so the seed update overlaps the next frame's tracking
    d2 = cpu_arm(CFG_NAME, 1, frames // 16, 1, 1, chain=args.chain, regime=args.seed_regime, dropin=True, two_threads=True)
    r2 = cpu_arm(CFG_NAME, 1, frames // 16, 1, 1, chain=args.chain, regime=args.seed_regime, two_threads=True)
    two = {"dropin_ms_per_frame": round(1e3 / d2["fps"], 4), "reference_ms_per_frame": round(1e3 / r2["fps"], 4),
           "speedup": round(d2["fps"] / r2["fps"], 3), "dropin_tracking_thread_p50_ms": round(d2["p50_ms"], 4),
           "reference_tracking_thread_p50_ms": round(r2["p50_ms"], 4), "cores": 2,
           "sample": "1 sequence x %d frames (+16 warm-up), tracking thread + depth-filter thread, no dropped frames; throughput over the whole "
                     "run incl. draining the filter's queue" % d2["frames"]}
    return {"impl": "dropin", "two_threads": two, "metric": "per-frame latency of the reference's own front-end loop with the hot-path TUs swapped for the B200 drop-in",
            "value": round(d["p50_ms"], 4), "unit": "ms", "n_gpus": 1, "steps": frames, "warmup": 16, "ms_per_step": round(d["mean_ms"], 4),
            "higher_is_better": False, "scaling": "none", "vs_baseline": None, "dtype": "u8 pixels / f32 photometric / f64 geometry", "data": "synthetic",
            "config": {"workload": "one C2 sequence (640x480, 4-level pyramid, %d map features, %d seeds), one host thread" % (cfg["n_features"], cfg["n_seeds"]),
                       "seed_regime": args.seed_regime, "step": "chain" if args.chain else "refine every map point of the keyframe"},
            "dropin": {"p50_ms": round(d["p50_ms"], 4), "p95_ms": round(d["p95_ms"], 4), "frames_per_s": round(d["fps"], 1), "per_operator_mean": d["per_operator"],
                       "tracked": d["tracked"]},
            "reference": {"p50_ms": round(r["p50_ms"], 4), "p95_ms": round(r["p95_ms"], 4), "frames_per_s": round(r["fps"], 1), "per_operator_mean": r["per_operator"],
                          "kind": r["kind"], "cores": 1, "tracked": r["tracked"]},
            "speedup_p50": round(r["p50_ms"] / d["p50_ms"], 3)}


_REAL_STDOUT = None


def claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1: park the real stdout, point fd 1 at stderr, and emit the one
    JSON line through the parked descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def main():
    args = parse_args()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = synth.CONFIGS[CFG_NAME]
    threads = os.cpu_count() or 1

    global METRIC
    if args.chain:
        METRIC = "front-end frames/s (pyramid + sparse align + reprojector + pose optimiser + seed update), batched C2 sequences"
    if args.impl in ("reference", "dropin"):
        # the reference's own CPU implementation of the path, all host threads, rank 0 only
        # (dropin: the SAME harness linked over the B200 drop-in: one sequence, one host thread, every operator call lands in CUDA)
        if rank != 0:
            return
        if args.impl == "dropin":
            line = dropin_line(args, cfg, threads)
            emit(json.dumps(line))
            return
        n = args.cpu_seqs or max(8, 4 * threads)
        r = cpu_arm(CFG_NAME, n, args.steps, args.warmup, threads, chain=args.chain, regime=args.seed_regime, kf_every=args.keyframe_every)
        line = {"impl": "reference", "metric": METRIC, "value": round(r["fps"], 2), "unit": "frames/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(r["seconds"] / args.steps * 1e3, 3),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8 pixels / f32 photometric / f64 geometry",
                "data": "synthetic",
                "config": {"workload": "C5: independent C2 sequences (640x480, 4-level pyramid, %d map features, %d seeds each); "
                                       "step = 1 frame of every sequence of the sample" % (cfg["n_features"], cfg["n_seeds"]),
                           "sequences_total": args.seqs, "sample_sequences": n, "frames_per_sequence_per_step": r["inner"],
                           "seed_regime": args.seed_regime, "keyframe_every": args.keyframe_every or None,
                           "step": "chain (reprojector + pose optimiser)" if args.chain else "refine every map point of the keyframe"},
                "cpu_baseline": {"value": round(r["fps"], 2), "unit": "frames/s", "cores": threads, "kind": r["kind"],
                                 "sample": "%d sequences x %d steps x %d frames (+%d warm-up steps), %d host threads, %.1f s wall"
                                           % (n, args.steps, r["inner"], args.warmup, threads, r["seconds"]),
                                 "per_frame_ms_on_a_loaded_core": {"p50": round(r["p50_ms"], 3), "p95": round(r["p95_ms"], 3)},
                                 "per_operator_mean": r["per_operator"]},
                "e2e": {"value": round(r["fps"], 2), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "tracked_mean": r["tracked"]}
        emit(json.dumps(line))
        return

    out, ctx, wl = run_b200(args, rank, world, local_rank)
    if rank == 0:
        from android_svo_b200 import capi
        if world == 1 and not args.no_widen:
            try:
                out["next_rows"] = widen_rows(ctx, capi, wl, cfg, out["roofline"]["peak"])
                if "pyramid_alone" in out["next_rows"]:
                    out["roofline_pyramid"]["alone"] = out["next_rows"].pop("pyramid_alone")
                if not args.no_cpu_baseline:
                    out["next_rows"]["cpu"] = widen_cpu(cfg)
            except Exception as e:   # pragma: no cover
                out["next_rows"] = {"error": repr(e)}
        if not args.no_latency:
            wl.close()
            out["latency"] = {}
            for name in ("C2", "C3", "C4"):
                try:
                    out["latency"][name] = latency_single(ctx, capi, name, chain=args.chain, regime=args.seed_regime)
                except Exception as e:   # pragma: no cover
                    out["latency"][name] = {"error": str(e)}
                if world == 1 and not args.no_cpu_baseline and "error" not in out["latency"][name]:
                    # the reference's per-frame latency on ONE host core, same sequence shape (its native single-stream mode): true
                    # per-frame p50 / p95 with the per-operator steady_clock split, for the -O2 build and the -O3 / AVX2 one
                    try:
                        out["latency"][name]["cpu_reference_1_thread"] = cpu_latency(name, chain=args.chain, regime=args.seed_regime,
                                                                                     frames=48 if name != "C4" else 32)
                        if name == "C2":
                            out["latency"][name]["cpu_reference_1_thread_o3"] = cpu_latency(name, chain=args.chain, regime=args.seed_regime, o3=True)
                        if not args.chain:
                            out["latency"][name]["cpu_reference_2_threads"] = cpu_two_threads(name, regime=args.seed_regime, frames=96 if name != "C4" else 48)
                    except Exception as e:   # pragma: no cover
                        out["latency"][name]["cpu_reference_1_thread"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            n = args.cpu_seqs or max(8, 4 * threads)
            r = cpu_arm(CFG_NAME, n, 10, 1, threads, chain=args.chain, regime=args.seed_regime, kf_every=args.keyframe_every)
            out["cpu_baseline"] = {"value": round(r["fps"], 2), "unit": "frames/s", "cores": threads, "kind": r["kind"],
                                   "sample": "%d sequences x 10 steps x %d frames (+1 warm-up step), %d host threads, %.1f s wall"
                                             % (n, r["inner"], threads, r["seconds"]),
                                   "per_operator_mean": r["per_operator"]}
        emit(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
