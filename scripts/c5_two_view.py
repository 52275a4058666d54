#!/usr/bin/env python
"""C5 with the second half of the reference's frame loop inside the lock step: tracker.step (:1713) and
find_E_ransac(K, step.prev_pts, step.cur_pts, 2500, 1e-3, 60) on that step's survivors (:1739, skipped without survivors,
:1715), for 64 independent 1080p sequences on ONE GPU (sfmgpu_multitracker with sfmgpu_multitracker_set_ransac).

bench.py's C5 shape (64 sequences x 64 frames, 2000 tracks, replenish below 818, 3 levels; frames synthesised and resident
on the device, the next step's frames prefetched while a step computes) timed in three arms, alternated within one process
after a warm-up:
    a  stage off (bench.py's C5 loop)
    b  stage on, early stop on (the default)
    c  stage on, early stop off (every hypothesis of every sequence solved and scored)
Prints one JSON line: ms per lock step, feature-tracks/s, the stage's device time (sfmgpu_stage_times_n[4], profiled pass),
launches per step, the fraction of sequences stopped early, and the reference-equivalent hyp*pts/s: sum over the sets that
reach find_E_ransac's scoring loop (>= 8 survivors) of iters x n, over the stage time - what the reference's loop evaluates;
with the early stop the device evaluates fewer.  Arms b and c must return identical results; the first and the last sequence
are checked against the CPU checker's find_E_ransac on the GPU's own survivors for the first 8 steps."""
import argparse
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
import bench  # noqa: E402  (C5 shape, seeds, K)
import sfmgpu  # noqa: E402

RS = dict(iters=2500, thr=1e-3, min_inliers=60, min_points=1)  # :1739 + the prev_pts.empty() guard (:1715)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sequences", type=int, default=bench.C5["sequences"])
    ap.add_argument("--frames", type=int, default=bench.C5["frames"])
    ap.add_argument("--rounds", type=int, default=3, help="timed passes per arm, alternated")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--check-steps", type=int, default=8)
    args = ap.parse_args()
    C5 = bench.C5
    W, H, S, T = C5["W"], C5["H"], args.sequences, args.frames
    K = bench.temple_K()
    ctx = sfmgpu.Context(0)
    info = gpu_info()
    store = ctx.frames(W, H, T * S, 1)  # frame t of sequence s at index t*S + s, as bench.py's C5
    for t in range(T):
        for q in range(S):
            store.synth(t * S + q, 1, bench.SEED0 + q, t)
    base, pitch, fstride = store.device_ptr(0)
    assert pitch == W and fstride == W * H
    step_bytes = S * W * H
    cfg = sfmgpu.lkcfg(max_tracks=C5["corners"], min_tracks=C5["min_tracks"], pyr_levels=bench.LEVELS)
    mt = ctx.multitracker(S, W, H, cfg)

    def arm(name):
        if name == "a":
            mt.set_ransac(None)
            return
        ctx.ransac_set_early_stop(name == "b")
        mt.set_ransac(K, **RS)

    def one_pass(record=False, fetch_first=0):
        """T lock steps; record: per step (survivor counts, status, best_n, inliers, R, t); fetch_first: survivors of the
        first steps too."""
        mt.reset()
        rec = []
        for t in range(T):
            nxt = base + (t + 1) * step_bytes if t + 1 < T else None
            out = mt.step_ptr(base if t == 0 else None, nxt, fetch=t < fetch_first)
            if record:
                n = np.array([len(o[0]) for o in out] if t < fetch_first else out, np.int64)
                rec.append((n, mt.ransac_results(), out if t < fetch_first else None))
        return rec

    for name in ("a", "b", "c"):
        arm(name)
        for _ in range(args.warmup):
            one_pass()
    ctx.sync()
    times = {k: [] for k in "abc"}
    launches = {k: [] for k in "abc"}
    tracks = {}
    for r in range(args.rounds):
        for name in ("abc", "bca", "cab")[r % 3]:
            arm(name)
            mt.ransac_early()
            l0 = ctx.launches()
            t0 = time.perf_counter()
            ctx.timer_start()
            one_pass()
            ms_dev = ctx.timer_stop()
            times[name].append(max(ms_dev, (time.perf_counter() - t0) * 1e3))  # every lock step synchronises: wall == device
            launches[name].append(ctx.launches() - l0)
            tracks[name] = mt.totals()[0]

    # stage device time: one profiled pass per arm (stage events cost host time: not part of the timed passes)
    stage = {}
    for name in "abc":
        arm(name)
        ctx.profile(True)
        ctx.stage_times()
        one_pass()
        st = ctx.stage_times()
        ctx.profile(False)
        stage[name] = st

    # results of b and c, and the work the reference's loop does on them
    recs, early = {}, {}
    for name in "bc":
        arm(name)
        mt.ransac_early()
        recs[name] = one_pass(record=True, fetch_first=args.check_steps)
        early[name] = mt.ransac_early()
    same = True
    for (nb, rb, _), (nc, rc, _) in zip(recs["b"], recs["c"]):
        sb, bb, ib, Rb, tb = rb
        sc, bc, ic, Rc, tc = rc
        ok = sb == 2
        same = same and np.array_equal(nb, nc) and np.array_equal(sb, sc) and np.array_equal(bb, bc)
        same = same and all(np.array_equal(x, y) for x, y in zip(ib, ic)) and np.array_equal(Rb[ok], Rc[ok]) and np.array_equal(tb[ok], tc[ok])
    scored_sets, hyp_pts, status_counts = 0, 0, [0, 0, 0]
    for n, (stt, _, _, _, _), _ in recs["b"]:
        for s in range(S):
            status_counts[int(stt[s])] += 1
            if stt[s] != 0 and n[s] >= 8:
                scored_sets += 1
                hyp_pts += RS["iters"] * int(n[s])

    # parity: first and last sequence, first check_steps steps, against find_E_ransac on the GPU's own survivors
    import oracle
    chk, kind = oracle.best()
    parity_ok, checked = True, 0
    t0 = time.perf_counter()
    for t, (n, (stt, bn, inl, R, tt), surv) in enumerate(recs["b"][:args.check_steps]):
        for s in sorted({0, S - 1}):
            prev, cur, _ = surv[s]
            checked += 1
            if len(prev) == 0:
                parity_ok = parity_ok and stt[s] == 0 and bn[s] == 0
                continue
            want = chk.find_E_ransac(np.asarray(K).reshape(3, 3), prev, cur, RS["iters"], RS["thr"], RS["min_inliers"])
            if want is None:
                parity_ok = parity_ok and stt[s] == 1
                continue
            parity_ok = parity_ok and stt[s] == 2 and bn[s] == len(want[2]) and np.array_equal(inl[s], want[2])
            parity_ok = parity_ok and np.abs(R[s] - want[0]).max() < 1e-6 and np.abs(tt[s] - want[1]).max() < 1e-6
    ref_s = time.perf_counter() - t0

    def arm_out(name):
        ms_pass = float(np.median(times[name]))
        out = {"ms_per_lock_step": ms_pass / T, "ms_per_pass": ms_pass, "ms_per_pass_all": times[name],
               "feature_tracks_per_s": tracks[name] / (ms_pass * 1e-3), "launches_per_step": launches[name][-1] / T,
               "stage_ms_per_step_profiled": stage[name]["ransac"] / T}
        if name != "a":
            out["stage_share_of_step"] = stage[name]["ransac"] / T / out["ms_per_lock_step"]
            out["reference_equivalent_hyp_pts_per_s"] = hyp_pts / (stage[name]["ransac"] * 1e-3)
        return out

    res = {"config": f"C5 + find_E_ransac(K, prev_pts, cur_pts, {RS['iters']}, {RS['thr']}, {RS['min_inliers']}) per sequence and step: "
                     f"{S} synthetic {W}x{H} sequences x {T} frames, {C5['corners']} tracks, replenish below {C5['min_tracks']}, "
                     f"{bench.LEVELS} levels, frames resident, one GPU",
           "gpu": info, "rounds": args.rounds, "warmup": args.warmup,
           "arms": {"a_stage_off": arm_out("a"), "b_stage_early_stop": arm_out("b"), "c_stage_full_scoring": arm_out("c")},
           "b_equals_c": bool(same),
           "early_stopped_fraction": early["b"] / max(scored_sets, 1), "early_stopped_sets": early["b"], "early_stopped_c": early["c"],
           "sets_reaching_scoring": scored_sets, "status_counts_skipped_none_ok": status_counts,
           "reference_equivalent_hyp_pts_per_pass": hyp_pts,
           "parity": {"ok": bool(parity_ok), "sequences": sorted({0, S - 1}), "steps": args.check_steps, "sets_checked": checked,
                      "checker": kind, "reference_s": ref_s,
                      "exact": ["status", "best_n", "inlier list"], "R_t_tol": 1e-6}}
    print(json.dumps(res))
    mt.close()
    store.close()
    ctx.close()
    return 0 if (same and parity_ok) else 1


if __name__ == "__main__":
    sys.exit(main())
