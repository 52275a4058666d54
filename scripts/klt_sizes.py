#!/usr/bin/env python
"""Tracker steps across an image-size change against same-size steps of the same tracker, in one process.

Cases: 1920x1080 -> 1280x720 with 2000 tracks, 3840x2160 -> 1920x1080 with 8000 tracks (3 levels, radius 5, 10 iterations,
min_tracks 0 so that no step replenishes and both kinds of step do the same tracking work).  Per round and case the tracker
is reset on frame 0 of the large size (not timed), then stepped once; the rounds alternate

    same:   large frame 0 -> large frame 1   (one-batch path: the lane-per-feature chain from 6000 tracks)
    resize: large frame 0 -> small frame 1   (two-geometry warp-per-feature KLT between the old and the new batch, plus the
                                              new batch's allocation and the old one's release)

Each step is timed with a host clock around sfmgpu_tracker_step, which returns after a stream synchronise; frames are host
images (synthesised on the device, downloaded once), so both kinds include the frame upload and pyramid build.  Prints one
JSON line per case (median / min ms per kind, survivors) and the card's name and power limit.

    python scripts/klt_sizes.py [--rounds 20] [--warmup 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
import sfmgpu  # noqa: E402

CASES = [((1920, 1080), (1280, 720), 2000), ((3840, 2160), (1920, 1080), 8000)]
SEED = 2024


def gpu_info(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1])}


def frames(ctx, w, h, n):
    f = ctx.frames(w, h, n, 1)
    f.synth(0, n, SEED, 0)
    out = [np.ascontiguousarray(f.download(i)) for i in range(n)]
    f.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    ctx = sfmgpu.Context(args.device)
    info = gpu_info(args.device)
    for (W, H), (w, h), nt in CASES:
        big, small = frames(ctx, W, H, 2), frames(ctx, w, h, 2)
        t = ctx.tracker(max_tracks=nt, min_tracks=0)
        t.set_size_change(True)
        ms = {"same": [], "resize": []}
        survivors = {}
        for r in range(args.warmup + args.rounds):
            for kind, img in (("same", big[1]), ("resize", small[1])):
                t.reset(big[0])
                ctx.sync()
                t0 = time.perf_counter()
                n = t.step(img, fetch=False)
                dt = (time.perf_counter() - t0) * 1e3
                if r >= args.warmup:
                    ms[kind].append(dt)
                survivors[kind] = n
        print(json.dumps({
            "case": f"{W}x{H}->{w}x{h}", "tracks": nt, "rounds": args.rounds,
            "same_ms_median": round(float(np.median(ms["same"])), 3), "same_ms_min": round(min(ms["same"]), 3),
            "resize_ms_median": round(float(np.median(ms["resize"])), 3), "resize_ms_min": round(min(ms["resize"]), 3),
            "survivors_same": survivors["same"], "survivors_resize": survivors["resize"], "gpu": info}))
        t.close()
    ctx.close()


if __name__ == "__main__":
    main()
