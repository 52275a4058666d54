#!/usr/bin/env python
"""Packed and resident input for the lock-step tracker over sequences of different image sizes (W2 / W3 of DESIGN §7, C5
settings: 2000 tracks, replenish below 818, LEVELS pyramid levels; --ransac adds find_E_ransac (:1739) with one camera per
sequence to every step).

    W2  64 sequences, 16 each of 1920x1080, 1440x1080, 1280x720, 640x480
    W3  64 sequences of 64 sizes (1920 - 16k) x (1080 - 8k)

One mixed tracker (sfmgpu_multitracker_create_sized), four arms, each a pass of reset + T steps, warmed up and alternated:

  host_raw       frames in pinned host memory, pipelined (the next step's frames travel while a step computes)
  packed_seq     one packed blob per sequence in pinned memory, sfmgpu_multitracker_step_packed pipelined
  packed_class   one step-major blob per size class (frame t of the i-th sequence of class c = blob frame t * n_c + i)
  resident       one frame batch per size class in HBM (pyramids built), sfmgpu_multitracker_step_frames_sized

Reported: card, power limit and SM clocks (same run); medians of ms per lock step and feature-tracks/s; launches per step;
the packed decode (sfmgpu_stage_times_n ms[6]) and the resident gather (ms[5]) per pass, from a profiled pass of their own;
blob bytes and ratio; the upload floors of one pass (pinned host-to-device copies of T steps' raw frames and of the per-class
blobs, CUDA events); and one flag per arm: every step's survivors, ids and counts (and the stage's results with --ransac)
byte-identical to host_raw.  The script exits non-zero if an arm differs.

    python scripts/multitracker_sized_input.py [--only W2,W3] [--ransac] [--rounds 5] [--frames 32] [--out path]"""
import argparse
import ctypes
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (C5 settings, levels)
import sfmgpu  # noqa: E402
from packed_input import copy_ms, gpu_info, pinned  # noqa: E402

RANSAC = (2500, 1e-3, 60, 1)
W2 = [c for c in [(1920, 1080), (1440, 1080), (1280, 720), (640, 480)] for _ in range(16)]
W3 = [(1920 - 16 * k, 1080 - 8 * k) for k in range(64)]


def K_of(w, h, s):
    a, b = w / 640.0, h / 480.0
    return np.array([[1520.4 * a, 0, 302.32 * a + s], [0, 1525.9 * a, 246.87 * b], [0, 0, 1.0]])


def workload(ctx, name, sizes, T, rounds, warmup, ransac, seed0):
    lib, vp = ctx.lib, ctypes.c_void_p
    S = len(sizes)
    cfg = sfmgpu.lkcfg(max_tracks=bench.C5["corners"], min_tracks=bench.C5["min_tracks"], pyr_levels=bench.LEVELS)
    classes = {}
    for s, wh in enumerate(sizes):
        classes.setdefault(wh, []).append(s)
    # per class: a store of T * n_c frames, frame t of its i-th sequence at t * n_c + i (pyramids built: the resident arm's
    # batch; level 0 packed step-major: the packed_class arm's blob)
    stores, where = {}, [None] * S
    for (w, h), members in classes.items():
        n = len(members)
        f = ctx.frames(w, h, T * n, bench.LEVELS)
        for i, s in enumerate(members):
            for t in range(T):
                f.synth(t * n + i, 1, seed0 + s, t)
            where[s] = (f, i, n)
        f.build_pyramid()
        stores[(w, h)] = f
    step_bytes = sum(w * h for w, h in sizes)
    host = ctx.pinned_empty((T, step_bytes), np.uint8)
    for t in range(T):
        o = 0
        for s, (w, h) in enumerate(sizes):
            f, i, n = where[s]
            host[t, o:o + w * h] = f.download(t * n + i, 0).reshape(-1)
            o += w * h

    def pinned_copy(a):
        b = ctx.pinned_empty(a.shape, np.uint8)
        b[:] = a
        return b

    class_blob = {}
    for wh, f in stores.items():
        class_blob[wh] = pinned_copy(f.pack(0, T * len(classes[wh]), out=np.empty(sfmgpu.pack_bound(*wh, T * len(classes[wh])), np.uint8)))
    seq_blobs = []
    tmp = {}
    for s, (w, h) in enumerate(sizes):
        if (w, h) not in tmp:
            tmp[(w, h)] = ctx.frames(w, h, T, 1)
        g = tmp[(w, h)]
        g.synth(0, T, seed0 + s, 0)
        seq_blobs.append(pinned_copy(g.pack(0, T, out=np.empty(sfmgpu.pack_bound(w, h, T), np.uint8))))
    for g in tmp.values():
        g.close()

    mt = ctx.multitracker(S, [w for w, _ in sizes], [h for _, h in sizes], cfg)
    if ransac:
        mt.set_ransac(np.stack([K_of(w, h, s) for s, (w, h) in enumerate(sizes)]), *RANSAC)
    n_out = mt.n.ctypes.data_as(vp)
    outs = [vp(a.ctypes.data) for a in (mt.prev, mt.cur, mt.ids)]

    def c_arrays(blobs):
        return (vp * S)(*[b.ctypes.data for b in blobs]), (ctypes.c_size_t * S)(*[b.nbytes for b in blobs])

    per_seq = c_arrays(seq_blobs) + ([np.full(S, t, np.int32) for t in range(T)],)
    per_class = c_arrays([class_blob[sizes[s]] for s in range(S)]) + (
        [np.array([t * where[s][2] + where[s][1] for s in range(S)], np.int32) for t in range(T)],)
    res_f = (vp * S)(*[where[s][0].h_ for s in range(S)])
    res_idx = [np.array([t * where[s][2] + where[s][1] for s in range(S)], np.int32) for t in range(T)]

    def raw_pass(fetch=None):
        mt.reset()
        for t in range(T):
            nxt = host[t + 1].ctypes.data if t + 1 < T else None
            o = outs if fetch else [None] * 3
            ctx._ck(lib.sfmgpu_multitracker_step_pipelined(ctx.h, mt.h_, vp(host[0].ctypes.data) if t == 0 else None,
                                                           vp(nxt) if nxt else None, *o, n_out))
            if fetch:
                fetch(t)
        return mt.totals()[0]

    def packed_pass(arrs, fetch=None):
        p, n, idx = arrs
        mt.reset()
        for t in range(T):
            cur = idx[t] if t == 0 else None
            nxt = idx[t + 1] if t + 1 < T else None
            o = outs if fetch else [None] * 3
            ctx._ck(lib.sfmgpu_multitracker_step_packed(ctx.h, mt.h_, p, n, None if cur is None else cur.ctypes.data_as(vp),
                                                        None if nxt is None else nxt.ctypes.data_as(vp), *o, n_out))
            if fetch:
                fetch(t)
        return mt.totals()[0]

    def resident_pass(fetch=None):
        mt.reset()
        for t in range(T):
            o = outs if fetch else [None] * 3
            ctx._ck(lib.sfmgpu_multitracker_step_frames_sized(ctx.h, mt.h_, res_f, res_idx[t].ctypes.data_as(vp), *o, n_out))
            if fetch:
                fetch(t)
        return mt.totals()[0]

    arms = {"host_raw": raw_pass, "packed_seq": lambda fetch=None: packed_pass(per_seq, fetch),
            "packed_class": lambda fetch=None: packed_pass(per_class, fetch), "resident": resident_pass}

    def digests(run):
        out = []

        def fetch(t):
            h = hashlib.sha256(mt.n.tobytes())
            for s in range(S):
                k = mt.n[s]
                h.update(mt.prev[s, :k].tobytes() + mt.cur[s, :k].tobytes() + mt.ids[s, :k].tobytes())
            if ransac:
                st, bn, inl, R, tt = mt.ransac_results()
                h.update(st.tobytes() + bn.tobytes())
                for s in range(S):
                    h.update(inl[s].tobytes())
                    if st[s] == 2:
                        h.update(R[s].tobytes() + tt[s].tobytes())
            out.append(h.hexdigest())
        run(fetch)
        return out

    for fn in arms.values():
        for _ in range(warmup):
            fn()
    want = digests(arms["host_raw"])
    identical = {k: digests(arms[k]) == want for k in arms if k != "host_raw"}

    def stage_ms(fn, stage):
        ms = (ctypes.c_float * 7)()
        ctx.sync()
        ctx._ck(lib.sfmgpu_stage_times_n(ctx.h, ms, 7))
        ctx.profile(True)
        fn()
        ctx.sync()
        ctx._ck(lib.sfmgpu_stage_times_n(ctx.h, ms, 7))
        ctx.profile(False)
        return float(ms[stage])

    decode = {k: [stage_ms(arms[k], 6) for _ in range(2)] for k in ("packed_seq", "packed_class")}
    gather = [stage_ms(arms["resident"], 5) for _ in range(2)]
    launches = {}
    for k, fn in arms.items():
        ctx.sync()
        n0 = ctx.launches()
        fn()
        ctx.sync()
        launches[k] = (ctx.launches() - n0) / T

    one = pinned((step_bytes,))
    one[:] = host[0]
    floor_raw = T * copy_ms(one)
    del one
    cb = pinned((sum(b.nbytes for b in class_blob.values()),))
    cb[:] = np.concatenate(list(class_blob.values()))
    floor_blob = copy_ms(cb)
    del cb

    times, tracks, names = {k: [] for k in arms}, {}, list(arms)
    for r in range(rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            ctx.sync()
            t0 = time.perf_counter()
            tracks[k] = arms[k]()
            ctx.sync()
            times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: float(np.median(v)) for k, v in times.items()}
    raw_bytes = T * step_bytes
    seq_bytes = int(sum(b.nbytes for b in seq_blobs))
    cls_bytes = int(sum(b.nbytes for b in class_blob.values()))
    rep = {
        "workload": f"{name}: {S} sequences of {len(classes)} sizes x {T} frames, {cfg.max_tracks} tracks, replenish below "
                    f"{cfg.min_tracks}, {bench.LEVELS} levels", "ransac": RANSAC if ransac else None,
        "raw_bytes": raw_bytes, "seq_blob_bytes": seq_bytes, "seq_ratio": raw_bytes / seq_bytes, "class_blob_bytes": cls_bytes,
        "class_ratio": raw_bytes / cls_bytes, "upload_floor_raw_ms": floor_raw, "upload_floor_blob_ms": floor_blob,
        "ms_per_step": {k: v / T for k, v in med.items()}, "ms_per_pass": med, "ms_all": times,
        "feature_tracks_per_s": {k: tracks[k] / (med[k] / 1e3) for k in arms}, "launches_per_step": launches,
        "decode_ms_per_pass": {k: float(np.median(v)) for k, v in decode.items()}, "gather_ms_per_pass": float(np.median(gather)),
        "identical_to_host_raw": identical,
    }
    mt.close()
    for f in stores.values():
        f.close()
    print(name, json.dumps(rep), file=sys.stderr, flush=True)
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="W2,W3")
    ap.add_argument("--ransac", action="store_true")
    ap.add_argument("--frames", type=int, default=32, help="steps per pass of W2")
    ap.add_argument("--frames-w3", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = sfmgpu.Context(0)
    out = {"gpu": gpu_info(0)}
    only = a.only.split(",")
    if "W2" in only:
        out["W2"] = workload(ctx, "W2", W2, a.frames, a.rounds, a.warmup, a.ransac, 20261501)
    if "W3" in only:
        out["W3"] = workload(ctx, "W3", W3, a.frames_w3, a.rounds, a.warmup, a.ransac, 20261601)
    out["gpu_after"] = gpu_info(0)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()
    if not all(v for w in ("W2", "W3") if w in out for v in out[w]["identical_to_host_raw"].values()):
        sys.exit("an arm's outputs differ from host_raw")


if __name__ == "__main__":
    main()
