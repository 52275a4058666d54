#!/usr/bin/env python
"""A/B of two library builds on the tracker objects: byte-for-byte results and the single-tracker step time.

The library is the one sfmgpu loads (SFMGPU_LIB selects another build of the same ABI), so each build runs in its own process:
    python scripts/ab_trackers.py --dump a.npz        (once per build)
    python scripts/ab_trackers.py --compare a.npz b.npz
    python scripts/ab_trackers.py --time              (one JSON line: ms per single-tracker step at 1080p)

--dump runs, on seeded synthetic frames (some sequences turn flat for two frames, so their tracks are lost and they are reset):
  * the single tracker through step and step_frames at 1080p, with the default configuration and a replenish-heavy one
    (min_tracks close to max_tracks, fb_thresh = -1: every track is dropped and the list refilled in every step);
  * the lock-step tracker (8 x 1080p, the C5 configuration) through raw, pipelined, packed and step_frames input, with and
    without the RANSAC stage;
  * sfmgpu_pair_frontend_segments with and without the RANSAC stage.
Every survivor, id, track list, total and RANSAC result is stored; --compare requires them to be identical."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
import sfmgpu  # noqa: E402

K = np.array([1520.4, 0, 302.32, 0, 1525.9, 246.87, 0, 0, 1.0])
RANSAC = (2500, 1e-3, 60, 1)
W, H = 1920, 1080
SINGLE = {"default": {}, "heavy": dict(max_tracks=2200, min_tracks=2150, fb_thresh=-1.0)}
C5 = dict(max_tracks=2000, min_tracks=818)


def synth_seq(ctx, seed, T, w, h, flat=()):
    """[T, h, w] of the device generator's frames; frames in `flat` are a constant grey."""
    f = ctx.frames(w, h, T, 1)
    f.synth(0, T, seed, 0)
    out = np.stack([np.full((h, w), 90, np.uint8) if t in flat else f.download(t) for t in range(T)])
    f.close()
    return out


def resident(ctx, imgs, levels=3):
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), levels)
    f.upload(0, np.ascontiguousarray(imgs))
    f.build_pyramid()
    return f


def put(out, key, vals):
    for i, v in enumerate(vals):
        out[f"{key}/{i}"] = np.asarray(v)


def single_arms(ctx, out):
    T = 10
    seqs = {"plain": synth_seq(ctx, 20261301, T, W, H), "flat": synth_seq(ctx, 20261302, T, W, H, flat=(4, 5))}
    for sname, imgs in seqs.items():
        f = resident(ctx, imgs)
        for cname, kw in SINGLE.items():
            for via in ("step", "step_frames"):
                tr = ctx.tracker(**kw)
                for t in range(T):
                    got = tr.step(imgs[t]) if via == "step" else tr.step_frames(f, t)
                    put(out, f"single/{sname}/{cname}/{via}/{t}", list(got) + list(tr.tracks()))
                put(out, f"single/{sname}/{cname}/{via}/totals", tr.totals())
                tr.close()
        f.close()


def multi_arms(ctx, out):
    S, T = 8, 8
    seqs = [synth_seq(ctx, 20261310 + s, T, W, H, flat=(3, 4) if s == 2 else ()) for s in range(S - 1)]
    seqs.append(np.full((T, H, W), 77, np.uint8))  # no corners at all: reset on every frame
    frames = np.ascontiguousarray(np.stack([np.stack([q[t] for q in seqs]) for t in range(T)]))  # [T, S, H, W]
    stack = ctx.pinned_empty(frames.shape, np.uint8)
    stack[:] = frames
    res = resident(ctx, frames.reshape(T * S, H, W))
    blobs = []
    for s in range(S):
        g = ctx.frames(W, H, T, 1)
        g.upload(0, np.ascontiguousarray(frames[:, s]))
        blobs.append(g.pack().copy())
        g.close()
    for ransac in (False, True):
        for via in ("raw", "pipelined", "packed", "step_frames"):
            mt = ctx.multitracker(S, W, H, **C5)
            if ransac:
                mt.set_ransac(K, *RANSAC)
            if via == "pipelined":
                mt.prefetch(stack[0])
            for t in range(T):
                if via == "raw":
                    got = mt.step(frames[t])
                elif via == "pipelined":
                    got = mt.step(None, next_imgs=stack[t + 1] if t + 1 < T else None)
                elif via == "packed":
                    got = mt.step_packed(blobs, np.full(S, t))
                else:
                    got = mt.step_frames(res, np.arange(S) + t * S)
                key = f"multi/{ransac}/{via}/{t}"
                put(out, key, [a for g_ in got for a in g_] + [a for s in range(S) for a in mt.tracks(s)])
                if ransac:
                    st, bn, inl, R, tr_ = mt.ransac_results()
                    put(out, key + "/ransac", [st, bn, R, tr_] + inl)
            put(out, f"multi/{ransac}/{via}/totals", mt.totals())
            mt.close()
    res.close()


def segment_arms(ctx, out):
    w, h, T, steps = 640, 480, 33, 8
    imgs = synth_seq(ctx, 20261320, T, w, h, flat=(11, 12))
    f = resident(ctx, imgs)
    cfg = sfmgpu.lkcfg(max_tracks=400, min_tracks=380)
    seg_first = [0, 8, 16, 24]
    P = len(seg_first) * steps
    for ransac in (False, True):
        p = ctx.pairs(P, 401)
        if ransac:
            p.set_ransac(K.reshape(3, 3), *RANSAC)
        p.run_segments(f, seg_first, steps, cfg)
        li, lj = np.zeros((P, p.cap, 2)), np.zeros((P, p.cap, 2))
        nk, nc = np.zeros(P, np.int32), np.zeros(P, np.int32)
        p.download_all(li, lj, nk, nc)
        ids = p.ids_download_all(P)
        vals = [nk, nc, p.totals()] + [a for r in range(P) for a in (li[r, :nk[r]], lj[r, :nk[r]], ids[r, :nk[r]])]
        if ransac:
            st, bn, inl, R, t = np.zeros(P, np.int32), np.zeros(P, np.int32), np.zeros((P, p.cap), np.int32), np.zeros((P, 9)), np.zeros((P, 3))
            p.ransac_download_all(st, bn, inl, R, t)
            vals += [st, bn, R, t] + [inl[r, :bn[r]] for r in range(P)]
        put(out, f"segments/{ransac}", vals)
        p.close()
    f.close()


def time_single(ctx, steps=2000, warm=20):
    """ms per host-fed and resident single-tracker step at 1080p with the default configuration (host clock; every step ends
    in a stream synchronisation)."""
    T = 16
    imgs = synth_seq(ctx, 20261330, T, W, H)
    f = resident(ctx, imgs)
    r = {}
    for via in ("step", "step_frames"):
        tr = ctx.tracker()
        for k in range(warm):
            tr.step(imgs[k % T]) if via == "step" else tr.step_frames(f, k % T)
        t0 = time.perf_counter()
        for k in range(warm, warm + steps):
            # forward and back through the sequence, so that consecutive frames stay neighbours
            i = k % (2 * T - 2)
            i = i if i < T else 2 * T - 2 - i
            tr.step(imgs[i], fetch=False) if via == "step" else tr.step_frames(f, i, fetch=False)
        r[f"{via}_ms"] = (time.perf_counter() - t0) * 1e3 / steps
        tr.close()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--dump", metavar="OUT.npz")
    ap.add_argument("--compare", nargs=2, metavar=("A.npz", "B.npz"))
    ap.add_argument("--time", action="store_true")
    args = ap.parse_args()
    if args.compare:
        a, b = (np.load(p) for p in args.compare)
        diff = sorted(set(a.files) ^ set(b.files)) + [k for k in a.files if k in b.files and not np.array_equal(a[k], b[k])]
        print(json.dumps({"arrays": len(a.files), "differ": len(diff), "first": diff[:10]}))
        sys.exit(1 if diff else 0)
    ctx = sfmgpu.Context(0)
    if args.dump:
        out = {}
        single_arms(ctx, out)
        multi_arms(ctx, out)
        segment_arms(ctx, out)
        np.savez(args.dump, **out)
        print(json.dumps({"lib": sfmgpu.LIB_PATH, "arrays": len(out)}))
    if args.time:
        print(json.dumps({"lib": sfmgpu.LIB_PATH, **time_single(ctx)}))
    ctx.close()


if __name__ == "__main__":
    main()
