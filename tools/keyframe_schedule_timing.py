"""Frames/s of device-memory tracker steps under two keyframe schedules, and the kernel times of one insertion.

bench.py's keyframe workload (4,096 C2 sequences, steady seed regime, a seed pool sized as bench.py sizes it) in two
variants that run alternately in one process:
  every_5th   every sequence takes a keyframe every 5 steps through svob200_tracker_add_keyframe (bench.py --keyframe-every 5)
  staggered   every step, the 1/5 of the sequences with b % 5 == k % 5 take one through svob200_tracker_add_keyframes with a mask
              in device memory (no host synchronisation)
Both insert as many keyframes per sequence.  Then torch.profiler records the kernels of three insertions at 1/5 selection and
three at full selection (add_keyframes, device memory) and reports each keyframe kernel's mean time per insertion: the
detector's should scale with the selected count.  Prints one JSON line with the card and its power limit.

  python tools/keyframe_schedule_timing.py [--seqs 4096] [--steps 50] [--warmup 10] [--rounds 3]
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


class Staggered:
    """device buffers of the staggered schedule: one mask per phase, the depth arguments"""

    def __init__(self, ctx, B):
        self.ctx = ctx
        self.masks = []
        for ph in range(KF_EVERY):
            m = (np.arange(B) % KF_EVERY == ph).astype(np.uint8)
            self.masks.append(ctx.dev_alloc(B)); ctx.dev_upload(self.masks[-1], m)
        self.full = ctx.dev_alloc(B); ctx.dev_upload(self.full, np.ones(B, np.uint8))
        self.dm = ctx.dev_alloc(4 * B); ctx.dev_upload(self.dm, np.full(B, bench.DEPTH_MEAN, np.float32))
        self.dn = ctx.dev_alloc(4 * B); ctx.dev_upload(self.dn, np.full(B, bench.DEPTH_MIN, np.float32))

    def close(self):
        for p in self.masks + [self.full, self.dm, self.dn]:
            self.ctx.dev_free(p)


def step_staggered(wl, st, order, k):
    a, b = order[k], order[k + 1]
    wl.trk.step_raw(wl.pool_dev[b], wl.cfg["w"], wl.in_dev[a][0], wl.in_dev[a][1], wl.stats_dev, capi.MEM_DEVICE)
    wl.trk.add_keyframes_raw(st.masks[k % KF_EVERY], st.dm, st.dn)


def timed(ctx, wl, step, warmup, steps):
    wl.reset()
    for k in range(warmup):
        step(k)
    ctx.sync()
    ctx.timer_start()
    for k in range(warmup, warmup + steps):
        step(k)
    ms = ctx.timer_stop_ms()
    return wl.B * steps / (ms * 1e-3)


def insertion_kernels(ctx, wl, st, order, mask, n=3):
    """mean device time per insertion of every kernel add_keyframes launches (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    wl.reset()
    wl.trk.step_raw(wl.pool_dev[order[1]], wl.cfg["w"], wl.in_dev[order[0]][0], wl.in_dev[order[0]][1], wl.stats_dev, capi.MEM_DEVICE)
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            wl.trk.add_keyframes_raw(mask, st.dm, st.dn)
        ctx.sync()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type is not None and str(e.device_type).endswith("CUDA") and e.count:
            name = e.key.replace("(anonymous namespace)::", "").split("(")[0].split("<")[0].strip()
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            out[name] = round(t / n / 1e3, 4)          # ms per insertion
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    ctx = capi.Context(0)
    cfg = synth.CONFIGS[bench.CFG_NAME]
    every = bench.GpuWorkload(ctx, capi, cfg, list(range(args.seqs)), kf_every=KF_EVERY)
    stag = bench.GpuWorkload(ctx, capi, cfg, list(range(args.seqs)), tex_dev=every.tex_dev, kf_every=KF_EVERY)
    st = Staggered(ctx, args.seqs)
    order = bench.ping_pong(len(bench.POOL_INDICES), 2 * (args.warmup + args.steps) + 8)
    fps = {"every_5th_all": [], "staggered_fifth": []}
    for _ in range(args.rounds):
        fps["every_5th_all"].append(timed(ctx, every, lambda k: every.step(order, k, capi.MEM_DEVICE), args.warmup, args.steps))
        fps["staggered_fifth"].append(timed(ctx, stag, lambda k: step_staggered(stag, st, order, k), args.warmup, args.steps))
    res = {"seqs": args.seqs, "steps": args.steps, "warmup": args.warmup, "keyframe_every": KF_EVERY,
           "frames_per_s": {k: [round(v) for v in vs] for k, vs in fps.items()},
           "add_keyframe_ms_host_wall_median": round(float(np.median(every.kf_ms)), 3)}
    if not args.no_profile:
        try:
            res["insertion_kernel_ms"] = {"fifth": insertion_kernels(ctx, stag, st, order, st.masks[0]),
                                          "all": insertion_kernels(ctx, stag, st, order, st.full)}
        except Exception as e:                             # (the frame rates above stand on their own)
            res["insertion_kernel_ms"] = {"error": repr(e)}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip()
    print(json.dumps(res))
    st.close()
    stag.close()
    every.close()
    ctx.close()


if __name__ == "__main__":
    main()
