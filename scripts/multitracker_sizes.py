#!/usr/bin/env python
"""The lock-step tracker over sequences of different image sizes: one mixed tracker against the trackers it replaces.

    W1  64 x 1920x1080 (the C5 shape): sfmgpu_multitracker_create against create_sized with 64 equal sizes
    W2  64 sequences, 16 each of 1920x1080, 1440x1080, 1280x720, 640x480: one mixed tracker against four same-size trackers
        stepped back to back
    W3  64 sequences of 64 sizes (1920 - 16k) x (1080 - 8k): one mixed tracker against 64 one-sequence trackers

Frames are generated on the device (sfmgpu_frames_synth) and handed to every step from device memory, back to back in
sequence order, so the numbers are the step's own work: uploads (device-to-device copies), pyramids, corners, KLT, compaction.
Every arm warms up once per shape, then the arms alternate within each of --rounds passes; reported are medians of:
ms per lock step, feature-tracks/s, launches per step, and (one profiled pass per arm) the KLT stage time (sfmgpu_stage_times_n
ms[2]) per million feature-tracks.  Outputs: W1 and W2 arms byte for byte (every tracker takes the lane chain in auto mode);
W3's one-sequence trackers take the warp-per-feature family, so the maximum position deviation and the id agreement are given.
Card, power limit and SM clock are read in the same run.  One JSON object on stdout (and --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
import sfmgpu  # noqa: E402

C5 = dict(max_tracks=2000, min_tracks=818)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q


def device_steps(ctx, sizes, T, seed0):
    """[T] device uint8 tensors: frame t of every sequence back to back (sequence s: its own synthetic sequence)."""
    per_seq = []
    for s, (w, h) in enumerate(sizes):
        f = ctx.frames(w, h, T, 1)
        f.synth(0, T, seed0 + s, 0)
        per_seq.append(torch.from_numpy(np.stack([f.download(t) for t in range(T)]).reshape(T, -1)).to("cuda:0"))
        f.close()
    steps = [torch.cat([p[t] for p in per_seq]).contiguous() for t in range(T)]
    del per_seq
    torch.cuda.synchronize()
    return steps


class Arm:
    """One or more trackers that together step all sequences; `parts` = (tracker, byte offset, bytes, first sequence)."""

    def __init__(self, ctx, name, groups, total_bytes):
        self.ctx, self.name, self.parts = ctx, name, []
        off = 0
        for sizes, sized in groups:
            S = len(sizes)
            ws, hs = [w for w, _ in sizes], [h for _, h in sizes]
            mt = ctx.multitracker(S, ws, hs, **C5) if sized else ctx.multitracker(S, ws[0], hs[0], **C5)
            nb = sum(w * h for w, h in sizes)
            self.parts.append((mt, off, nb))
            off += nb
        assert off == total_bytes

    def run(self, steps, fetch=False):
        """One pass (reset + every step); returns (seconds, launches, feature-tracks, survivors per step if fetch)."""
        for mt, _, _ in self.parts:
            mt.reset()
        self.ctx.sync()
        n0, tr0 = self.ctx.launches(), sum(mt.totals()[0] for mt, _, _ in self.parts)
        outs = []
        t0 = time.perf_counter()
        for st in steps:
            base = st.data_ptr()
            got = []
            for mt, off, _ in self.parts:
                r = mt.step_ptr(base + off, None, fetch=fetch)
                if fetch:
                    got += r
            outs.append(got)
        self.ctx.sync()
        dt = time.perf_counter() - t0
        tr = sum(mt.totals()[0] for mt, _, _ in self.parts) - tr0
        return dt, self.ctx.launches() - n0, tr, outs

    def klt_per_mtracks(self, steps):
        self.ctx.profile(True)
        _, _, tr, _ = self.run(steps)
        ms = self.ctx.stage_times()["klt"]
        self.ctx.profile(False)
        return ms / tr * 1e6

    def close(self):
        for mt, _, _ in self.parts:
            mt.close()


def compare(a, b):
    """(identical, max |position difference|, ids equal) over every step and sequence."""
    same, dev, ids = True, 0.0, True
    for sa, sb in zip(a, b):
        for (pa, ca, ia), (pb, cb, ib) in zip(sa, sb):
            if not (np.array_equal(pa, pb) and np.array_equal(ca, cb) and np.array_equal(ia, ib)):
                same = False
            if np.array_equal(ia, ib):
                dev = max(dev, float(np.nanmax(np.abs(pa - pb), initial=0.0)), float(np.nanmax(np.abs(ca - cb), initial=0.0)))
            else:
                ids = False
    return same, dev, ids


def workload(ctx, name, sizes, arms, T, rounds, seed):
    steps = device_steps(ctx, sizes, T, seed)
    total = sum(w * h for w, h in sizes)
    objs = [Arm(ctx, n, g, total) for n, g in arms]
    outs = [o.run(steps, fetch=True)[3] for o in objs]  # warm-up and the outputs
    res = {o.name: {"s": [], "launches": 0, "tracks": 0} for o in objs}
    for _ in range(rounds):
        for o in objs:
            dt, nl, tr, _ = o.run(steps)
            r = res[o.name]
            r["s"].append(dt)
            r["launches"], r["tracks"] = nl, tr
    rep = {"sequences": len(sizes), "steps": T, "arms": {}}
    for o in objs:
        r = res[o.name]
        med = float(np.median(r["s"]))
        rep["arms"][o.name] = {"ms_per_step": 1e3 * med / T, "feature_tracks_per_s": r["tracks"] / med,
                               "launches_per_step": r["launches"] / T, "klt_ms_per_mtracks": o.klt_per_mtracks(steps),
                               "passes_ms": [1e3 * x for x in r["s"]]}
    same, dev, ids = compare(outs[0], outs[1])
    rep["outputs_identical"], rep["max_position_dev_px"], rep["ids_equal"] = same, dev, ids
    for o in objs:
        o.close()
    del steps
    torch.cuda.empty_cache()
    print(name, json.dumps(rep), file=sys.stderr, flush=True)
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=32, help="steps per pass of W1 and W2")
    ap.add_argument("--frames-w3", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default="W1,W2,W3")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = sfmgpu.Context(0)
    out = {"card": card(), "config": C5}
    only = a.only.split(",")
    if "W1" in only:
        sz = [(1920, 1080)] * 64
        out["W1"] = workload(ctx, "W1", sz, [("create", [(sz, False)]), ("create_sized", [(sz, True)])], a.frames, a.rounds, 20261401)
    if "W2" in only:
        cls = [(1920, 1080), (1440, 1080), (1280, 720), (640, 480)]
        sz = [c for c in cls for _ in range(16)]
        out["W2"] = workload(ctx, "W2", sz, [("mixed", [(sz, True)]), ("per_size", [([c] * 16, False) for c in cls])], a.frames, a.rounds,
                             20261501)
    if "W3" in only:
        sz = [(1920 - 16 * k, 1080 - 8 * k) for k in range(64)]
        out["W3"] = workload(ctx, "W3", sz, [("mixed", [(sz, True)]), ("single", [([c], False) for c in sz])], a.frames_w3, a.rounds,
                             20261601)
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
