"""Frames/s of device-memory tracker steps with and without a point pool (svob200_tracker_set_point_pool).

bench.py's keyframe workload (4,096 C2 sequences, steady seed regime, a keyframe every 5 steps: --keyframe-every 5) in two
variants that run alternately in one process: the tracker as bench.py builds it, and the same tracker with a point pool of
(set_keyframe points + 64) slots per sequence, whose converged seeds become map points.  The pool variant passes a last_px
entry per slot: the map points' projections, and an off-image pixel for the slots that start empty.  Prints one JSON line.

  python tools/point_pool_timing.py [--seqs 4096] [--steps 50] [--warmup 10] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True
import bench  # noqa: E402
from android_svo_b200 import capi, synth  # noqa: E402

KF_EVERY = 5
EXTRA_SLOTS = 64


def with_point_pool(ctx, wl, capacity):
    """replace the workload's tracker by the same tracker with a point pool, and its per-step pixels by one entry per slot"""
    cfg, B, N, S = wl.cfg, wl.B, wl.cfg["n_features"], wl.cfg["n_seeds"]
    wl.trk.close()
    trk = capi.Tracker(ctx, wl.cam, B, cfg["n_levels"], cfg["max_level"], cfg["min_level"], cfg["n_pyr"], 100.0, bench.DEPTH_MEAN, bench.DEPTH_MIN, 1)
    sc, st = bench.frontend.DETECT[bench.CFG_NAME][2:]
    n_cells = -(-cfg["w"] // sc) * -(-cfg["h"] // sc)           # as bench.GpuWorkload sizes the seed pool
    trk.set_seed_pool(S + (bench.KF_RING - 1) * n_cells, bench.KF_RING, bench.KF_MAX_N_KFS, 3)
    trk.set_detector(sc, cfg["n_pyr"], st)
    trk.set_point_pool(capacity)
    kf = wl.kf
    trk.set_keyframe(wl.kf_host, wl.poses[:, 0], np.arange(B + 1) * N, kf["kf_px"].reshape(-1, 2), kf["kf_level"].reshape(-1),
                     kf["pt_world"].reshape(-1, 3), np.arange(B + 1) * S, kf["seed_px"].reshape(-1, 2), kf["seed_level"].reshape(-1))
    P = trk.P // B
    in_dev = []
    for k, (dT, dp) in enumerate(wl.in_dev):
        lp = np.full((B, P, 2), -100.0)
        lp[:, :N] = bench.project_many(cfg, np.ascontiguousarray(wl.poses[:, 1 + k]), kf["pt_world"]).reshape(B, N, 2)
        d = ctx.dev_alloc(lp.nbytes)
        ctx.dev_upload(d, lp)
        ctx.dev_free(dp)
        in_dev.append((dT, d))
    wl.trk, wl.in_dev = trk, in_dev
    return P


def timed(ctx, wl, order, warmup, steps):
    wl.reset()
    for k in range(warmup):
        wl.step(order, k, capi.MEM_DEVICE)
    ctx.sync()
    ctx.timer_start()
    for k in range(warmup, warmup + steps):
        wl.step(order, k, capi.MEM_DEVICE)
    ms = ctx.timer_stop_ms()
    return wl.B * steps / (ms * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    ctx = capi.Context(0)
    cfg = synth.CONFIGS[bench.CFG_NAME]
    base = bench.GpuWorkload(ctx, capi, cfg, list(range(args.seqs)), kf_every=KF_EVERY)
    pool = bench.GpuWorkload(ctx, capi, cfg, list(range(args.seqs)), tex_dev=base.tex_dev, kf_every=KF_EVERY)
    P = with_point_pool(ctx, pool, cfg["n_features"] + EXTRA_SLOTS)
    order = bench.ping_pong(len(bench.POOL_INDICES), 2 * (args.warmup + args.steps) + 8)
    fps = {"no_pool": [], "point_pool": []}
    for _ in range(args.rounds):
        fps["no_pool"].append(timed(ctx, base, order, args.warmup, args.steps))
        fps["point_pool"].append(timed(ctx, pool, order, args.warmup, args.steps))
    _, ty, _, created, dropped = pool.trk.points()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    print(json.dumps({"seqs": args.seqs, "steps": args.steps, "warmup": args.warmup, "keyframe_every": KF_EVERY, "slots_per_sequence": P,
                      "frames_per_s": {k: [round(v) for v in vs] for k, vs in fps.items()},
                      "overhead_pct_of_medians": round(100.0 * (1 - np.median(fps["point_pool"]) / np.median(fps["no_pool"])), 2),
                      "points": {"candidates": int((ty == capi.POINT_CANDIDATE).sum()), "map_points": int((ty >= capi.POINT_UNKNOWN).sum()),
                                 "empty": int((ty == capi.POINT_DELETED).sum()), "created": int(created.sum()), "dropped": int(dropped.sum())},
                      "gpu": q.stdout.strip()}))
    pool.close()
    base.close()
    ctx.close()


if __name__ == "__main__":
    main()
