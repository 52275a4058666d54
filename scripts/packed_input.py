#!/usr/bin/env python
"""Packed frame input on the C3 and C2 shapes (bench.py's frames, seed, corners and RANSAC stage): the streaming front end fed
raw u8 frames (sfmgpu_pair_frontend_host) against the same call fed a packed blob of the same frames
(sfmgpu_pair_frontend_host_packed), alternated in one process after a warm-up, next to the resident step (pyramids + the pair
front end on resident frames: the compute bound of both host-fed calls).

Reported per workload: card and power limit; blob bytes and compression ratio; device encode time (sfmgpu_frames_pack, host
clock around the call, which ends when the blob is in host memory); decode kernel time of one pass over all frames
(sfmgpu_stage_times_n ms[6], CUDA events); the upload floors, pure pinned host-to-device copies of the raw frames and of the
blob (torch copy, CUDA events); the three arms' times (host clock around calls that end in a synchronise; medians of --rounds
passes); and whether the two host-fed arms' outputs (survivors, counts, RANSAC status, counts, inlier lists, R, t) are byte
identical.  The bytes to upload fall by the ratio; what is left of the packed call over the resident step is decode + the
pipeline fill (first upload, last chunk) - compare the two floors and the decode time with that gap.

    python scripts/packed_input.py [--workloads c3,c2] [--rounds 3] [--frames N]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload shapes, seed, K, RANSAC settings)
import sfmgpu  # noqa: E402


def gpu_info(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}


def copy_ms(src_np, reps=3):
    """Median ms of a pure host-to-device copy of a pinned numpy array (one cudaMemcpyAsync through torch)."""
    import torch
    src = torch.from_numpy(src_np.reshape(-1))
    assert src.is_pinned()
    dst = torch.empty(src.numel(), dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src, non_blocking=True)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    del dst
    torch.cuda.empty_cache()
    return float(np.median(ts[1:]))


def pinned(shape):
    """Page-locked host array (torch's pinned allocator, so that torch's copies see it as pinned too)."""
    import torch
    return torch.empty(int(np.prod(shape)), dtype=torch.uint8, pin_memory=True).numpy().reshape(shape)


def outputs(ctx, P, cap):
    return dict(li=ctx.pinned_empty((P, cap, 2), np.float64), lj=ctx.pinned_empty((P, cap, 2), np.float64),
                nk=ctx.pinned_empty((P,), np.int32), nc=ctx.pinned_empty((P,), np.int32), status=ctx.pinned_empty((P,), np.int32),
                best_n=ctx.pinned_empty((P,), np.int32), inliers=ctx.pinned_empty((P, cap), np.int32),
                R=ctx.pinned_empty((P, 9), np.float64), t=ctx.pinned_empty((P, 3), np.float64))


def same_outputs(a, b):
    """Byte comparison of what the call defines: counts and statuses, survivors up to n_kept, inliers up to best_n, R and t of
    pairs with a pose."""
    if any(a[x].tobytes() != b[x].tobytes() for x in ("nk", "nc", "status", "best_n")):
        return False
    for k in range(len(a["nk"])):
        n, m = a["nk"][k], max(a["best_n"][k], 0)
        if a["li"][k, :n].tobytes() != b["li"][k, :n].tobytes() or a["lj"][k, :n].tobytes() != b["lj"][k, :n].tobytes():
            return False
        if a["inliers"][k, :m].tobytes() != b["inliers"][k, :m].tobytes():
            return False
        if a["status"][k] == 2 and (a["R"][k].tobytes() != b["R"][k].tobytes() or a["t"][k].tobytes() != b["t"][k].tobytes()):
            return False
    return True


def run_workload(ctx, key, nframes, rounds, warmup):
    wl = bench.WORKLOADS[key]
    W, H, cap, n = wl["W"], wl["H"], wl["corners"], nframes or wl["frames"]
    P = n - 1
    cfg = sfmgpu.lkcfg(max_tracks=cap, pyr_levels=bench.LEVELS)
    fr = ctx.frames(W, H, n, bench.LEVELS)
    fr.synth(0, n, bench.SEED0, 0)
    ctx.sync()
    host = pinned((n, H, W))
    for j in range(n):
        host[j] = fr.download(j, 0)

    # device encode (the blob lands in pageable memory sized by the bound, then moves to pinned memory of its own size)
    room = np.empty(sfmgpu.pack_bound(W, H, n), np.uint8)
    t0 = time.perf_counter()
    packed = fr.pack(0, n, out=room)
    enc_ms = (time.perf_counter() - t0) * 1e3
    blob = pinned(packed.shape)
    blob[:] = packed
    del packed, room

    # decode kernel time per pass (profiled upload_packed over all frames)
    dec = []
    for _ in range(3):
        ctx.profile(True)
        fr.upload_packed(0, blob)
        ms = (ctypes.c_float * 7)()
        ctx._ck(ctx.lib.sfmgpu_stage_times_n(ctx.h, ms, 7))
        ctx.profile(False)
        dec.append(ms[6])
    assert all(np.array_equal(fr.download(j, 0), host[j]) for j in (0, n // 2, n - 1)), "decoded frames differ"

    floor_raw, floor_blob = copy_ms(host), copy_ms(blob)

    pr, pp = ctx.pairs(P, cap), ctx.pairs(P, cap)
    out_r, out_p = outputs(ctx, P, cap), outputs(ctx, P, cap)
    for p, o in ((pr, out_r), (pp, out_p)):
        p.set_ransac(bench.temple_K(), **bench.RANSAC)
        p.ransac_host_outputs(o["status"], o["best_n"], o["inliers"], o["R"], o["t"])

    def raw():
        pr.run_host(fr, host, cfg, out_r["li"], out_r["lj"], out_r["nk"], out_r["nc"])

    def pk():
        pp.run_host_packed(fr, blob, n, cfg, out_p["li"], out_p["lj"], out_p["nk"], out_p["nc"])

    def resident():
        fr.build_pyramid(0, n)
        pr.run(fr, 0, P, cfg)

    arms = {"host_raw": raw, "host_packed": pk, "resident": resident}
    for f in arms.values():
        for _ in range(warmup):
            f()
    times = {k: [] for k in arms}
    names = list(arms)
    identical = True
    for r in range(rounds):
        for k in names[r % 3:] + names[:r % 3]:
            ctx.sync()
            t0 = time.perf_counter()
            arms[k]()
            ctx.sync()
            times[k].append((time.perf_counter() - t0) * 1e3)
            if k == "host_packed":  # the raw arm's outputs are from an earlier pass over the same frames
                identical &= same_outputs(out_r, out_p)
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {
        "workload": wl["name"], "frames": n, "width": W, "height": H, "max_corners": cap, "ransac": bench.RANSAC,
        "raw_bytes": int(host.nbytes), "blob_bytes": int(blob.nbytes), "ratio": host.nbytes / blob.nbytes,
        "encode_ms": enc_ms, "decode_kernel_ms_per_pass": float(np.median(dec)), "decode_passes_ms": dec,
        "upload_floor_raw_ms": floor_raw, "upload_floor_blob_ms": floor_blob,
        "raw_gbps": host.nbytes / floor_raw / 1e6, "blob_gbps": blob.nbytes / floor_blob / 1e6,
        "ms": med, "ms_all": times,
        "packed_over_resident": med["host_packed"] / med["resident"], "raw_over_resident": med["host_raw"] / med["resident"],
        "outputs_byte_identical": bool(identical),
    }
    for a in list(out_r.values()) + list(out_p.values()):
        ctx.pinned_free(a)
    pr.close()
    pp.close()
    fr.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c2")
    ap.add_argument("--frames", type=int, default=0, help="override the workloads' frame counts (0: bench.py's)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the report as JSON to this path")
    args = ap.parse_args()
    ctx = sfmgpu.Context(0)
    report = {"gpu": gpu_info(0), "results": []}
    for key in args.workloads.split(","):
        r = run_workload(ctx, key, args.frames, args.rounds, args.warmup)
        print(json.dumps(r), flush=True)
        report["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(report, fh, indent=1)
    print(json.dumps(report["gpu"]))
    ctx.close()
    if not all(r["outputs_byte_identical"] for r in report["results"]):
        sys.exit("host_raw and host_packed outputs differ")


if __name__ == "__main__":
    main()
