#!/usr/bin/env python
"""Batched loop closure on one GPU: the device-resident descriptor search and the two-view unit over explicit frame pairs.

Search: a bank of N descriptors (global_desc_32, :1100-1122) of 1080p synth frames computed on the device, every keyframe k
searched against slots [0, k - gap) (:1823-1831) in one sfmgpu_descs_search call, against the same work as N
sfmgpu_desc_search calls (host arrays: the bank's prefix is uploaded on every call).  Reports the kernel time
(torch.profiler, CUDA activities), the call time (device events), dot products/s, FP32 operations/s and their share of the
non-FMA FP32 issue rate (SMs x 128 lanes x max SM clock), all computed from shapes.  Both arms must agree bit for bit.

List front end: P random non-adjacent pairs among F resident 1080p synth frames through sfmgpu_pair_frontend_list with the
RANSAC stage at the loop-closure settings (max_tracks 1200, find_E_ransac(K, li, lj, 4000, 2e-3, 80), li.size() >= 120,
:1836-1857), against P consecutive pairs through sfmgpu_pair_frontend with the stage pipeline off, and the list call on the
same consecutive pairs; arms alternated after a warm-up.  The list call on consecutive pairs must equal the consecutive
call byte for byte.  The gather's share comes from a separate profiled pass (sfmgpu_stage_times_n[5]).

Prints the card name and power limit with the numbers, and one JSON line at the end."""
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
import sfmgpu  # noqa: E402

K = np.array([1520.4, 0, 302.32, 0, 1525.9, 246.87, 0, 0, 1.0])
W, H, SEED = 1920, 1080, 20261020


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}


def kernel_ms(fn, name, reps):
    """Mean device time of kernels whose name contains `name` over `reps` calls of fn, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = 0.0
    for e in prof.key_averages():
        if name in e.key:
            tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return tot / 1e3 / reps if tot else None


def search_arm(ctx, info, n, gap, reps):
    f = ctx.frames(W, H, n, 1)
    f.synth(0, n, SEED, 0)
    bank = ctx.descs(n)
    bank.compute(f, 0, n)
    f.close()
    qs = np.arange(n, dtype=np.int32)
    ns = np.maximum(qs - gap, 0).astype(np.int32)
    dots = int(ns.sum())
    flops = 2 * 1024 * dots
    bid, bs, _ = bank.search(qs, ns)  # warm-up
    ms_call = []
    for _ in range(reps):
        ctx.timer_start()
        bank.search(qs, ns)
        ms_call.append(ctx.timer_stop())
    try:
        ms_kernel = kernel_ms(lambda: bank.search(qs, ns), "desc_search_kernel", reps)
    except Exception as e:  # noqa: BLE001  (the profiler is optional: report the event time alone)
        print(f"torch.profiler unavailable: {e}", file=sys.stderr)
        ms_kernel = None
    # the same work as n single-query calls on host arrays
    host = bank.download()
    ctx.desc_search(host[:1], host[0], 1)
    t0 = time.perf_counter()
    single = [ctx.desc_search(host[:ns[k]], host[k], int(ns[k]))[:2] for k in range(n)]
    ms_single = (time.perf_counter() - t0) * 1e3
    same = all(single[k][0] == bid[k] and np.float32(single[k][1]).tobytes() == np.float32(bs[k]).tobytes() for k in range(n))
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lanes = sms * 128
    issue = lanes * info["sm_max_mhz"] * 1e6  # non-FMA FP32 operations/s
    t_k = ms_kernel if ms_kernel else float(np.median(ms_call))
    return {
        "bank": n, "gap": gap, "dot_products": dots, "fp32_ops": flops,
        "kernel_ms": ms_kernel, "call_ms_median": float(np.median(ms_call)),
        "dots_per_s": dots / (t_k * 1e-3), "fp32_ops_per_s": flops / (t_k * 1e-3),
        "share_of_nonfma_fp32_issue": flops / (t_k * 1e-3) / issue, "sms": sms,
        "per_query_calls_ms": ms_single, "speedup_vs_per_query": ms_single / t_k,
        "candidates": int((bid >= 0).sum()), "arms_equal": bool(same),
    }


def stage_times6(ctx):
    ms = (C.c_float * 6)()
    ctx._ck(ctx.lib.sfmgpu_stage_times_n(ctx.h, ms, 6))
    return list(ms)


def outputs(pairs, n):
    cap = pairs.cap
    li, lj = np.zeros((n, cap, 2)), np.zeros((n, cap, 2))
    nk, nc = np.zeros(n, np.int32), np.zeros(n, np.int32)
    pairs.download_all(li, lj, nk, nc)
    st, bn = np.zeros(n, np.int32), np.zeros(n, np.int32)
    inl, R, t = np.zeros((n, cap), np.int32), np.zeros((n, 9)), np.zeros((n, 3))
    pairs.ransac_download_all(st, bn, inl, R, t)
    out = [nk, nc, np.array(pairs.totals()), st, bn]
    for k in range(n):
        out += [li[k, :nk[k]], lj[k, :nk[k]], inl[k, :max(bn[k], 0)]]
    ok = st == 2
    return out + [R[ok], t[ok]]


def list_arm(ctx, nframes, npairs, rounds, seed):
    f = ctx.frames(W, H, nframes, 3)
    f.synth(0, nframes, SEED, 0)
    f.build_pyramid()
    rng = np.random.default_rng(seed)
    fa, fb = [], []
    while len(fa) < npairs:
        a, b = (int(v) for v in rng.integers(0, nframes, 2))
        if abs(a - b) >= 2:
            fa.append(a)
            fb.append(b)
    fa, fb = np.array(fa, np.int32), np.array(fb, np.int32)
    ca = np.arange(npairs, dtype=np.int32)
    cfg = sfmgpu.lkcfg(max_tracks=1200)
    pairs = ctx.pairs(npairs, 1200)
    pairs.set_ransac(K, 4000, 2e-3, 80, 120)
    ctx.pipeline_set(0)
    arms = {
        "list_random": lambda: pairs.run_list(f, fa, fb, cfg),
        "consecutive": lambda: pairs.run(f, 0, npairs, cfg),
        "list_consecutive": lambda: pairs.run_list(f, ca, ca + 1, cfg),
    }
    for fn in arms.values():  # warm-up
        fn()
    pairs.run(f, 0, npairs, cfg)
    want = outputs(pairs, npairs)
    pairs.run_list(f, ca, ca + 1, cfg)
    got = outputs(pairs, npairs)
    same = len(want) == len(got) and all(np.asarray(a).tobytes() == np.asarray(b).tobytes() for a, b in zip(want, got))
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ctx.timer_start()
            fn()
            ms[k].append(ctx.timer_stop())
    pairs.run_list(f, fa, fb, cfg)
    rnd = outputs(pairs, npairs)
    st = rnd[3]
    # profiled passes: stage times of the random-pair list call and of the consecutive call
    ctx.profile(True)
    stage_times6(ctx)
    ctx.timer_start()
    pairs.run_list(f, fa, fb, cfg)
    ms_prof = ctx.timer_stop()
    st6 = stage_times6(ctx)
    pairs.run(f, 0, npairs, cfg)
    st6_consec = stage_times6(ctx)
    ctx.profile(False)
    names = ("corner_score", "corner_select", "klt", "compact", "ransac", "gather")
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return {
        "frames": nframes, "pairs": npairs,
        "ms_per_pair": {k: v / npairs for k, v in med.items()},
        "call_ms_median": med,
        "list_random_over_consecutive": med["list_random"] / med["consecutive"],
        "list_consecutive_over_consecutive": med["list_consecutive"] / med["consecutive"],
        "random_pairs_corners_kept_lkiters": [int(v) for v in rnd[2]],
        "consecutive_corners_kept_lkiters": [int(v) for v in want[2]],
        "random_pairs_status_counts": {s: int((st == i).sum()) for i, s in enumerate(("skipped", "none", "ok"))},
        "profiled_call_ms": ms_prof,
        "stage_ms": dict(zip(names, st6)),
        "stage_ms_consecutive": dict(zip(names, st6_consec)),
        "gather_share_of_call": st6[5] / ms_prof,
        "list_equals_consecutive": bool(same),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bank", type=int, default=2000)
    ap.add_argument("--gap", type=int, default=6)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    info = gpu_info()
    ctx = sfmgpu.Context(0)
    print(f"GPU: {info['name']}, power limit {info['power_limit_w']:.0f} W, SM max {info['sm_max_mhz']:.0f} MHz")
    s = search_arm(ctx, info, args.bank, args.gap, args.reps)
    km = f"{s['kernel_ms']:.3f} ms" if s["kernel_ms"] else "not measured"
    print(f"search: {s['dot_products']} dot products, kernel {km}, call {s['call_ms_median']:.3f} ms, "
          f"{s['dots_per_s'] / 1e9:.2f} G dots/s, {s['fp32_ops_per_s'] / 1e12:.2f} T FP32 ops/s = "
          f"{100 * s['share_of_nonfma_fp32_issue']:.1f} % of the non-FMA FP32 issue rate; {args.bank} single-query calls "
          f"{s['per_query_calls_ms']:.1f} ms ({s['speedup_vs_per_query']:.0f}x); arms equal: {s['arms_equal']}")
    l = list_arm(ctx, args.frames, args.pairs, args.rounds, args.seed)
    print(f"list front end: ms/pair {json.dumps({k: round(v, 4) for k, v in l['ms_per_pair'].items()})}, random list / "
          f"consecutive {l['list_random_over_consecutive']:.3f}, consecutive list / consecutive "
          f"{l['list_consecutive_over_consecutive']:.3f}, gather {100 * l['gather_share_of_call']:.1f} % of the call; "
          f"list == consecutive: {l['list_equals_consecutive']}")
    print(json.dumps({"gpu": info, "search": s, "list": l}))
    ctx.close()
    if not (s["arms_equal"] and l["list_equals_consecutive"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
