#!/usr/bin/env python
"""Segment mode on the C3 shape: ONE resident sequence of 2000 synthetic 3840x2160 frames (bench.py's C3 seed, 3 levels) cut
into G segments per GPU (sfmgpu_sched_segment_shard), each a fresh KLTTracker (max_tracks 8000, replenish below 3272 = C5's
818/2000 ratio) with find_E_ransac(K, prev, cur, 2500, 1e-3, 60) on every step's survivors (:1739), run by
sfmgpu_pair_frontend_segments.  For contrast, pair mode (sfmgpu_pair_frontend, detection on every frame) on the same resident
frames with the same RANSAC settings, alternated with the segment arms in one process after a warm-up.  The two workloads
differ: segment mode detects corners only at resets and replenishment, pair mode on every frame.

Per arm: ms per call (CUDA events around the call, which ends in a synchronise), feature-tracks/s = sum of n_corners over all
rows / time, the RANSAC stage's and the frame gather's device times (one profiled call, sfmgpu_stage_times_n ms[4], ms[5]), the
gather's modelled bytes (every level of every slot's frame read and written once per lock step) and its share of the call,
and the sets stopped early.  Parity: rank 0 gathers the rows, track ids and stage results of all ranks (NCCL for N > 1, a
local copy for one GPU) and checks the first and last segment of every rank against the CPU checker's KLTTracker and
find_E_ransac for their first --check-steps steps.

    python scripts/segment_mode.py --segments 32,64
    torchrun --nproc_per_node N scripts/segment_mode.py --segments 32,64     (each rank synthesises only its frames)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (C3 shape, seed, K)
import sfmgpu  # noqa: E402
from sfmgpu import sched, synth  # noqa: E402

RS = (2500, 1e-3, 60, 1)  # :1739 + the prev_pts.empty() guard (:1715)


def gpu_info(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", default="32,64", help="segments per GPU, comma separated (one arm each)")
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3, help="timed calls per arm, alternated")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--check-steps", type=int, default=3)
    args = ap.parse_args()
    C3 = bench.WORKLOADS["c3"]
    W, H, T, NT = C3["W"], C3["H"], args.frames, C3["corners"]
    MIN_T = round(NT * 818 / 2000)
    ROWS = NT + 1
    K = np.asarray(bench.temple_K(), np.float64).reshape(3, 3)
    Gs = [int(g) for g in args.segments.split(",")]

    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    ctx = sfmgpu.Context(dev)
    lib = ctx.lib
    info = gpu_info(dev)
    uid = (C.c_uint8 * 128)()
    if world > 1:
        if rank == 0 and lib.sfmgpu_sched_unique_id(uid) != 0:
            raise RuntimeError("sfmgpu_sched_unique_id failed")
        obj = [bytes(uid)]
        dist.broadcast_object_list(obj, src=0)
        uid = (C.c_uint8 * 128).from_buffer_copy(obj[0])
    sch = C.c_void_p()
    ctx._ck(lib.sfmgpu_sched_create(ctx.h, world, rank, uid if world > 1 else None, None, C.byref(sch)))

    # frames this rank needs: the union over the arms
    shards = {G: sched.segment_shard(T, G * world, world, rank) for G in Gs}
    f0 = min(s[4] for s in shards.values())
    f1 = max(s[5] for s in shards.values())
    t0 = time.perf_counter()
    fr = ctx.frames(W, H, f1 - f0, bench.LEVELS)
    fr.synth(0, f1 - f0, bench.SEED0, f0)
    fr.build_pyramid()
    ctx.sync()
    synth_s = time.perf_counter() - t0
    cfg = sfmgpu.lkcfg(max_tracks=NT, min_tracks=MIN_T, pyr_levels=bench.LEVELS)
    pm_cfg = sfmgpu.lkcfg(max_tracks=NT, pyr_levels=bench.LEVELS)
    level_bytes = sum(fr.device_ptr(l)[2] for l in range(bench.LEVELS))

    arms = {}
    for G in Gs:
        L, a, b, first, _, _ = shards[G]
        p = ctx.pairs(max((b - a) * L, 1), ROWS)
        p.set_ransac(K, *RS)
        arms[f"seg{G}"] = dict(kind="seg", G=G, L=L, a=a, b=b, first=first, local=first[a:b] - f0, pairs=p)
    npm = f1 - f0 - 1
    pm = ctx.pairs(npm, NT)
    pm.set_ransac(K, *RS)
    arms["pair"] = dict(kind="pair", pairs=pm)

    def run(arm):
        if arm["kind"] == "seg":
            arm["pairs"].run_segments(fr, arm["local"], arm["L"], cfg)
        else:
            arm["pairs"].run(fr, 0, npm, pm_cfg)

    for arm in arms.values():
        for _ in range(args.warmup):
            run(arm)
    names = list(arms)
    times = {k: [] for k in names}
    tracks, early = {}, {}
    for r in range(args.rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            arms[k]["pairs"].ransac_early()
            ctx.timer_start()
            run(arms[k])
            times[k].append(ctx.timer_stop())
            tracks[k] = arms[k]["pairs"].totals()[0]
            early[k] = arms[k]["pairs"].ransac_early()
    stage = {}
    for k in names:  # stage events cost host time: a separate profiled call
        ctx.profile(True)
        ms6 = (C.c_float * 6)()
        lib.sfmgpu_stage_times_n(ctx.h, ms6, 6)
        ctx.timer_start()
        run(arms[k])
        total = ctx.timer_stop()
        ctx._ck(lib.sfmgpu_stage_times_n(ctx.h, ms6, 6))
        ctx.profile(False)
        stage[k] = dict(ransac_ms=ms6[4], gather_ms=ms6[5], call_ms_profiled=total)

    out = {}
    for k in names:
        arm, ms = arms[k], float(np.median(times[k]))
        o = {"ms_per_call": ms, "ms_all": times[k], "feature_tracks": tracks[k], "feature_tracks_per_s": tracks[k] / (ms * 1e-3),
             "ransac_stage_ms": stage[k]["ransac_ms"], "early_stopped_sets": early[k]}
        if arm["kind"] == "seg":
            nseg = arm["b"] - arm["a"]
            gbytes = 2 * level_bytes * nseg * (arm["L"] + 1)
            o.update(segments=nseg, steps=arm["L"], rows=nseg * arm["L"], gather_ms=stage[k]["gather_ms"],
                     gather_share=stage[k]["gather_ms"] / stage[k]["call_ms_profiled"], gather_bytes_model=gbytes,
                     gather_gb_per_s=gbytes / max(stage[k]["gather_ms"], 1e-9) * 1e-6)
        else:
            o.update(pairs=npm)
        out[k] = o

    # parity through the gathers: every arm's rows, ids and stage results on rank 0; first and last segment of every rank
    parity = {}
    import oracle
    chk, kind = oracle.best()
    for G in Gs:
        arm = arms[f"seg{G}"]
        run(arm)
        L, first, P = arm["L"], arm["first"], G * world * arm["L"]
        root = rank == 0
        nk = np.zeros(P, np.int32) if root else None
        nc = np.zeros(P, np.int32) if root else None
        st = np.zeros(P, np.int32) if root else None
        bn = np.zeros(P, np.int32) if root else None
        li = np.zeros((P, ROWS, 2)) if root else None
        lj = np.zeros((P, ROWS, 2)) if root else None
        inl = np.zeros((P, ROWS), np.int32) if root else None
        R, t = (np.zeros((P, 9)), np.zeros((P, 3))) if root else (None, None)
        ids = np.zeros((P, ROWS), np.int32) if root else None
        ptr = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)  # noqa: E731
        ctx._ck(lib.sfmgpu_sched_gather_pairs(ctx.h, sch, arm["pairs"].h_, P, 0, 1, ptr(li), ptr(lj), ptr(nk), ptr(nc), ptr(st), ptr(bn),
                                              ptr(inl), ptr(R), ptr(t)))
        ctx._ck(lib.sfmgpu_sched_gather_pair_ids(ctx.h, sch, arm["pairs"].h_, P, 0, ptr(ids)))
        if not root:
            continue
        ok, checked, pose_dev, t_ref = True, [], 0.0, time.perf_counter()
        sample = sorted({j for r_ in range(world) for j in (G * r_, G * r_ + G - 1)})
        for j in sample:
            s0 = int(first[j])
            tr = chk.tracker(max_tracks=NT, min_tracks=MIN_T)
            tr.step(synth.frame(bench.SEED0, s0, W, H))
            for k in range(min(args.check_steps, L)):
                r_ = j * L + k
                n_in = len(tr.tracks()[1])
                prev, cur, tid = tr.step(synth.frame(bench.SEED0, s0 + k + 1, W, H))
                n = nk[r_]
                bad = []  # what differs from the checker
                if not (nc[r_] == n_in and n == len(tid) and np.array_equal(ids[r_, :n], tid)):
                    bad.append(f"counts/ids {nc[r_]}/{n_in} {n}/{len(tid)}")
                elif n and max(np.abs(li[r_, :n] - prev).max(), np.abs(lj[r_, :n] - cur).max()) > 1e-3:
                    bad.append("positions")
                want = chk.find_E_ransac(K, prev, cur, *RS[:3]) if len(prev) else None
                if len(prev) == 0 or want is None:
                    if st[r_] != (0 if len(prev) == 0 else 1):
                        bad.append(f"status {st[r_]}")
                elif not (st[r_] == 2 and bn[r_] == len(want[2]) and np.array_equal(inl[r_, :bn[r_]], want[2])):
                    bad.append(f"status/inliers {st[r_]} {bn[r_]}/{len(want[2])}")
                else:  # bench.py's pose tolerance for this shape (device solver + device pose tail, thousands of inliers)
                    dev = max(np.abs(R[r_] - np.ravel(want[0])).max(), np.abs(t[r_] - np.ravel(want[1])).max())
                    pose_dev = max(pose_dev, float(dev))
                    if dev > bench.POSE_TOL:
                        bad.append(f"pose {dev:.2e}")
                ok = ok and not bad
                checked.append([j, k + 1, int(n), int(st[r_])] + bad)
        parity[f"seg{G}"] = {"ok": ok, "checked_segment_step_kept_status": checked, "checker": kind,
                             "exact": ["ids", "n_corners", "n_kept", "status", "best_n", "inlier list"], "pos_tol_px": 1e-3,
                             "pose_tol": bench.POSE_TOL, "max_pose_dev": pose_dev, "reference_s": time.perf_counter() - t_ref}

    rank_out = {"rank": rank, "frames": [f0, f1], "synth_s": synth_s, "arms": out}
    per_rank = [None] * world
    if world > 1:
        dist.all_gather_object(per_rank, rank_out)
    else:
        per_rank = [rank_out]
    if rank == 0:
        res = {"config": f"C3 as segments: {T} synthetic {W}x{H} frames resident (seed {bench.SEED0}), {bench.LEVELS} levels, "
                         f"max_tracks {NT}, min_tracks {MIN_T}, find_E_ransac(K, prev, cur, {RS[0]}, {RS[1]}, {RS[2]}) per step; "
                         f"pair mode on the same frames with the same RANSAC settings (detection on every frame: another workload)",
               "gpu": info, "world": world, "rounds": args.rounds, "warmup": args.warmup, "ranks": per_rank, "parity": parity}
        print(json.dumps(res))
    lib.sfmgpu_sched_destroy(ctx.h, sch)
    for arm in arms.values():
        arm["pairs"].close()
    fr.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0 if all(v["ok"] for v in parity.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
