#!/usr/bin/env python
"""Packed frame input for the lock-step tracker on bench.py's C5 shape (64 independent 1080p sequences x 64 frames, seeds
SEED0 + s, 2000 tracks, replenish below 818, LEVELS pyramid levels; --ransac adds find_E_ransac (:1739) to every step).
Four pipelined arms (reset + T steps, the next frames travelling while a step computes), alternated in one process after a
warm-up:

  resident       source frames in HBM (the device pointers bench.py times as `value`)
  host_raw       source frames in pinned host memory (bench.py's `e2e`)
  packed_step    one step-major packed blob in pinned memory (Frames.pack of the same store: frame t of sequence s = blob
                 frame t*S + s, one copy per step), sfmgpu_multitracker_step_packed
  packed_seq     64 per-sequence blobs (64 copies per step)

Reported: card, power limit and SM max clock (same run); blob bytes and ratio; the upload floors of one pass (pure pinned
host-to-device copies, CUDA events: T copies of one step's raw frames, and the whole step-major blob; both from torch's pinned
allocator, the memory torch's copy recognises as page-locked); the decode kernel time per pass (sfmgpu_stage_times_n
ms[6] of a profiled pass, on the copy stream beside the step's kernels, and of a pass of plain steps where nothing overlaps
it); the median ms per pass and feature-tracks/s of each arm.  Every step's survivors and ids of all sequences (and the stage
results with --ransac) of both packed arms are compared byte for byte with the raw arm's; the script exits non-zero if they
differ.

    python scripts/c5_packed.py [--ransac] [--rounds 5] [--sequences 64] [--frames 64] [--out path]"""
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
import bench  # noqa: E402  (C5 shape, seed, levels)
import sfmgpu  # noqa: E402
from packed_input import copy_ms, gpu_info, pinned  # noqa: E402

RANSAC = (2500, 1e-3, 60, 1)  # find_E_ransac(K, prev, cur, 2500, 1e-3, 60) (:1739), skipped without survivors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ransac", action="store_true", help="run the :1739 RANSAC stage inside every step")
    ap.add_argument("--sequences", type=int, default=bench.C5["sequences"])
    ap.add_argument("--frames", type=int, default=bench.C5["frames"])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the report as JSON to this path")
    args = ap.parse_args()
    W, H, S, T = bench.C5["W"], bench.C5["H"], args.sequences, args.frames
    ctx = sfmgpu.Context(0)
    lib = ctx.lib
    cfg = sfmgpu.lkcfg(max_tracks=bench.C5["corners"], min_tracks=bench.C5["min_tracks"], pyr_levels=bench.LEVELS)

    store = ctx.frames(W, H, T * S, 1)  # bench.py's store: frame t of sequence s at index t*S + s
    for t in range(T):
        for q in range(S):
            store.synth(t * S + q, 1, bench.SEED0 + q, t)
    base, pitch, fstride = store.device_ptr(0)
    assert pitch == W and fstride == W * H
    host = ctx.pinned_empty((T, S, H, W), np.uint8)
    for k in range(T * S):
        host.reshape(T * S, H, W)[k] = store.download(k, 0)
    packed = store.pack(0, T * S, out=np.empty(sfmgpu.pack_bound(W, H, T * S), np.uint8))
    blob = ctx.pinned_empty(packed.shape, np.uint8)
    blob[:] = packed
    del packed
    seq_blobs = []
    f = ctx.frames(W, H, T, 1)
    for q in range(S):
        f.synth(0, T, bench.SEED0 + q, 0)  # the same frames as the store's sequence q
        p = f.pack(0, T, out=np.empty(sfmgpu.pack_bound(W, H, T), np.uint8))
        b = ctx.pinned_empty(p.shape, np.uint8)
        b[:] = p
        seq_blobs.append(b)
    f.close()
    store_raw = host.nbytes

    mt = ctx.multitracker(S, W, H, cfg)
    if args.ransac:
        mt.set_ransac(bench.temple_K(), *RANSAC)
    step_bytes = S * W * H
    n_out = mt.n.ctypes.data_as(ctypes.c_void_p)
    vp = ctypes.c_void_p

    def c_arrays(blobs):
        return (vp * S)(*[b.ctypes.data for b in blobs]), (ctypes.c_size_t * S)(*[b.nbytes for b in blobs])

    step_major = c_arrays([blob] * S) + ([np.ascontiguousarray(t * S + np.arange(S), np.int32) for t in range(T)],)
    per_seq = c_arrays(seq_blobs) + ([np.full(S, t, np.int32) for t in range(T)],)
    outs = [vp(a.ctypes.data) for a in (mt.prev, mt.cur, mt.ids)]

    def ptr_pass(src, fetch=None):
        mt.reset()
        for t in range(T):
            nxt = src + (t + 1) * step_bytes if t + 1 < T else None
            o = outs if fetch else [None] * 3
            ctx._ck(lib.sfmgpu_multitracker_step_pipelined(ctx.h, mt.h_, vp(src + t * step_bytes) if t == 0 else None,
                                                           vp(nxt) if nxt else None, *o, n_out))
            if fetch:
                fetch(t)
        return mt.totals()[0]

    def packed_pass(arrs, fetch=None, pipelined=True):
        p, n, idx = arrs
        mt.reset()
        for t in range(T):
            cur = idx[t] if (t == 0 or not pipelined) else None
            nxt = idx[t + 1] if (pipelined and t + 1 < T) else None
            o = outs if fetch else [None] * 3
            ctx._ck(lib.sfmgpu_multitracker_step_packed(ctx.h, mt.h_, p, n, None if cur is None else cur.ctypes.data_as(vp),
                                                        None if nxt is None else nxt.ctypes.data_as(vp), *o, n_out))
            if fetch:
                fetch(t)
        return mt.totals()[0]

    def digests(run):
        """sha256 per step of every sequence's survivors, ids and counts (and the stage's results)."""
        out = []

        def fetch(t):
            h = hashlib.sha256(mt.n.tobytes())
            for s in range(S):
                k = mt.n[s]
                h.update(mt.prev[s, :k].tobytes())
                h.update(mt.cur[s, :k].tobytes())
                h.update(mt.ids[s, :k].tobytes())
            if args.ransac:
                st, bn, inl, R, tt = mt.ransac_results()
                h.update(st.tobytes() + bn.tobytes())
                for s in range(S):
                    h.update(inl[s].tobytes())
                    if st[s] == 2:
                        h.update(R[s].tobytes() + tt[s].tobytes())
            out.append(h.hexdigest())
        run(fetch)
        return out

    arms = {
        "resident": lambda fetch=None: ptr_pass(base, fetch),
        "host_raw": lambda fetch=None: ptr_pass(host.ctypes.data, fetch),
        "packed_step": lambda fetch=None: packed_pass(step_major, fetch),
        "packed_seq": lambda fetch=None: packed_pass(per_seq, fetch),
    }
    for fn in arms.values():
        for _ in range(args.warmup):
            fn()

    # byte comparison of every step against the raw arm
    want = digests(arms["host_raw"])
    identical = {k: digests(arms[k]) == want for k in ("resident", "packed_step", "packed_seq")}
    identical["packed_step_plain"] = digests(lambda fetch: packed_pass(step_major, fetch, pipelined=False)) == want

    # decode kernel time per pass: beside the step's kernels (pipelined), and alone (plain steps)
    def decode_ms(fn):
        ms = (ctypes.c_float * 7)()
        ctx.sync()
        ctx._ck(lib.sfmgpu_stage_times_n(ctx.h, ms, 7))
        ctx.profile(True)
        fn()
        ctx.sync()
        ctx._ck(lib.sfmgpu_stage_times_n(ctx.h, ms, 7))
        ctx.profile(False)
        return float(ms[6])

    dec_pipe = [decode_ms(arms["packed_step"]) for _ in range(2)]
    dec_plain = [decode_ms(lambda: packed_pass(step_major, pipelined=False)) for _ in range(2)]

    one_step = pinned((S, H, W))
    one_step[:] = host[0]
    floor_raw = T * copy_ms(one_step)
    del one_step
    blob_t = pinned(blob.shape)
    blob_t[:] = blob
    floor_blob = copy_ms(blob_t)
    del blob_t

    times = {k: [] for k in arms}
    tracks = {}
    names = list(arms)
    for r in range(args.rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            ctx.sync()
            t0 = time.perf_counter()
            tracks[k] = arms[k]()
            ctx.sync()
            times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: float(np.median(v)) for k, v in times.items()}
    seq_bytes = int(sum(b.nbytes for b in seq_blobs))
    res = {
        "workload": f"C5 packed: {S} sequences x {T} frames of {W}x{H}, {cfg.max_tracks} tracks, replenish below {cfg.min_tracks}",
        "gpu": gpu_info(0), "ransac": RANSAC if args.ransac else None,
        "raw_bytes": int(store_raw), "blob_bytes": int(blob.nbytes), "ratio": store_raw / blob.nbytes,
        "seq_blob_bytes": seq_bytes, "seq_ratio": store_raw / seq_bytes,
        "upload_floor_raw_ms": floor_raw, "upload_floor_blob_ms": floor_blob,
        "raw_gbps": store_raw / floor_raw / 1e6, "blob_gbps": blob.nbytes / floor_blob / 1e6,
        "decode_kernel_ms_per_pass_pipelined": float(np.median(dec_pipe)), "decode_kernel_ms_per_pass_alone": float(np.median(dec_plain)),
        "decode_passes_ms": {"pipelined": dec_pipe, "alone": dec_plain},
        "ms": med, "ms_all": times,
        "feature_tracks_per_s": {k: tracks[k] / (med[k] / 1e3) for k in arms},
        "track_steps_per_pass": tracks,
        "identical_to_host_raw": identical,
    }
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)
    mt.close()
    store.close()
    ctx.close()
    if not all(identical.values()):
        sys.exit(f"outputs differ from the raw arm: {identical}")


if __name__ == "__main__":
    main()
