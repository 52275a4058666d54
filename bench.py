#!/usr/bin/env python
"""bench.py — the front-end hot path on synthetic sequences, one JSON line on stdout.

Workload (BASELINE.json configs[2], "C3", the configuration north_star names for scaling): ONE synthetic 3840x2160
2,000-frame sequence (seed 20261018, integer generator of sfmgpu/synth.py), 8,000 corners per frame, run as the
reference's stateless two-view unit (cpp/src/templering_sfm.cpp:1836-1857) over all 1,999 frame pairs:
    3-level pyramid -> Shi-Tomasi + exact std::sort order + greedy NMS -> forward + backward pyramidal LK -> fb filter ->
    if (li.size() >= 120) find_E_ransac(K, li, lj, 4000, 2e-3, 80)   (sampling, 8-point solver, Sampson scoring, pose)
One "step" = one pass over the whole sequence.  With N GPUs the PAIRS are sharded: rank g owns a contiguous block of
pairs plus one halo frame (SURVEY.md §8e mode 1), total work fixed -> "scaling": "strong"; no data-path collective, the
results (tracks, counts, inlier sets, poses) are gathered to rank 0 over NCCL at the end of an end-to-end step.
`--workload c2` runs configs[1] (1080p x 1000 frames, 2000 corners) the same way; at N=1 a shorter C2 measurement is
attached to the line as "c2".

metric  : KLT feature-tracks/s (1 feature-track = fwd + bwd track_one + fb test of one corner, SURVEY.md §8d) for the
          whole unit incl. its RANSAC stage; the RANSAC half of BASELINE.json's metric (hyp x pts / s, config C4) is
          reported under "ransac".
value   : frames resident in HBM, CUDA events on the library's stream, max over ranks.  The library's default path: the
          RANSAC stage stops solving / scoring a pair - exactly - once one of its first 128 hypotheses explains all of its
          points (DESIGN.md §4); "ransac_early_stop" reports the fraction of pairs stopped and the same step with the stop
          off (every hypothesis of every pair solved and scored, as the reference does) as "full_scoring".
e2e     : the same step through the C ABI with HOST (pinned) frames: H2D of the frames and D2H of tracks, inlier sets and
          poses inside the timed region (N > 1: plus the NCCL gather to rank 0, which then reads everything back).
parity_in_bench : the reference (oracle/_ref) runs the same unit on sample pairs of the same frames on the host; corner
          counts, survivor counts, li, RANSAC status / inlier lists must be identical, lj within 1e-3 px.
--impl reference : the reference's own CPU implementation of the unit on all host cores, bounded sample per step.
--dump-outputs DIR : the results of the last timed resident step as .npy files (dump_outputs); the inputs depend on the
          arguments only, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))

WORKLOADS = {
    "c3": dict(name="C3", W=3840, H=2160, frames=2000, corners=8000),
    "c2": dict(name="C2", W=1920, H=1080, frames=1000, corners=2000),
}
LEVELS = 3
SEED0 = 20261018
RANSAC = dict(iters=4000, thr=2e-3, min_inliers=80, min_points=120)  # the unit's own call, :1855-1857
METRIC = "KLT feature-tracks/sec (+ RANSAC hyp*pts/sec under 'ransac')"
UNIT = "feature-tracks/s"
B_KLT = 2092.0      # algorithmic bytes per feature-track (SURVEY.md §8d)
F_KLT_IT = 5045.0   # algorithmic FP64 flop per LK iteration (SURVEY.md §8d)
F_RS = 35.0         # flop per hyp x pt (SURVEY.md §8d)
RS_N, RS_H = 10000, 65536
KLT_TOL = 1e-3      # px, north_star's tolerance for tracked positions
POSE_TOL = 1e-4     # R, t entries through the device solver + device pose tail (inlier lists are compared bit for bit)


def temple_K():
    return np.array([1520.4, 0, 302.32, 0, 1525.9, 246.87, 0, 0, 1.0])


def shard_range(n_items, world, rank):
    """The scheduler's block partition (sfmgpu_sched_shard of the C ABI, through sfmgpu/sched.py)."""
    from sfmgpu import sched
    return sched.shard_range(n_items, world, rank)


def workload_cfg(wl, n_gpus, nframes):
    return {
        "workload": f"{wl['name']}: ONE synthetic {wl['W']}x{wl['H']} {nframes}-frame sequence, two-view unit over all {nframes - 1} pairs "
                    f"(pyramid L={LEVELS} + Shi-Tomasi/NMS {wl['corners']} corners/frame + fwd/bwd KLT r=5 iters=10 + fb<1.0 + "
                    f"find_E_ransac({RANSAC['iters']}, {RANSAC['thr']}, {RANSAC['min_inliers']}) per pair with >= {RANSAC['min_points']} survivors)",
        "frames": nframes, "pairs": nframes - 1, "width": wl["W"], "height": wl["H"], "max_corners": wl["corners"],
        "pyr_levels": LEVELS, "ransac": RANSAC,
        "sharding": f"pair blocks + one halo frame per rank x{n_gpus} (no data-path collective; NCCL gather of results to rank 0)",
        "l2_policy": f"inputs ({wl['W'] * wl['H'] * nframes / n_gpus / 1e9:.2f} GB of frames per GPU) exceed the 126 MB L2; no explicit flush needed",
        "ransac_workload": f"C4: {RS_H} hypotheses x {RS_N} correspondences, thr 1e-3, hypotheses = the seeded sampler's octets through the 8-point solver",
    }


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.p, self.lines = index, None, []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_near_gpu(index):
    """Pin this rank (and therefore its first-touch pinned allocations) to the CPUs NVML reports as local to its GPU.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def profile_metrics():
    """ncu-derived numbers of the committed captures (profiles/*_metrics.json): static evidence, labelled as such."""
    out = {}
    for fn in ("r2_metrics.json", "r1_metrics.json"):
        try:
            with open(os.path.join(ROOT, "profiles", fn)) as fh:
                m = json.load(fh)
        except Exception:
            continue
        for name, d in m.items():
            for short in ("klt_quad_kernel", "score_tile_kernel<2>", "radix_sort_frame_kernel", "nms_kernel", "ransac_count_kernel", "pyr_down_kernel",
                          "eight_point_kernel"):
                if short in name and short not in out:
                    out[short] = dict(d, source=f"profiles/{fn}")
    return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback (of fallback)"


def c4_points(n):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import TEMPLE_K, two_view_scene
    pi, pj = two_view_scene(n)
    Kinv = np.linalg.inv(TEMPLE_K)

    def norm(p):
        hp = np.concatenate([p, np.ones((len(p), 1))], 1) @ Kinv.T
        return np.ascontiguousarray(hp[:, :2] / hp[:, 2:3])
    return norm(pi), norm(pj)


def host_threads():
    return max(1, min(len(os.sched_getaffinity(0)), 64))


# ---------------------------------------------------------------------------------------------------------------
def run_reference(args, wl, rank):
    """The reference's CPU implementation of the unit on all host cores (rank 0 only): every step runs `threads` pairs of the
    same sequence (one per host thread) through detection, KLT, fb filter and find_E_ransac."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    chk, kind = oracle.best()
    gen = oracle.port()
    threads = host_threads()
    if args.workload == "c5":
        return run_reference_c5(args, chk, gen, kind, threads)
    frames = gen.synth_frames(SEED0, 0, threads + 1, wl["W"], wl["H"], threads=threads)
    K = temple_K()
    times, tracks = [], 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        tracks, _ = chk.two_view_mt(frames, wl["corners"], threads, K=K, rs_iters=RANSAC["iters"], rs_thr=RANSAC["thr"],
                                    rs_min_inliers=RANSAC["min_inliers"], min_points=RANSAC["min_points"], detail=False)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times)) if times else float("nan")
    val = tracks / (ms * 1e-3) if times else 0.0
    xi, xj = c4_points(RS_N)
    Hs = 64 * threads
    E = chk.ransac_hypotheses(xi, xj, 64)[0]
    E = np.ascontiguousarray(np.tile(E, (threads, 1)))
    t0 = time.perf_counter()
    chk.ransac_score_mt(xi, xj, E, 1e-3, threads)
    rs = Hs * RS_N / (time.perf_counter() - t0)
    sample = (f"{threads} pairs of the {wl['name']} sequence per step (one per host thread), {tracks} feature-tracks, front end + "
              f"find_E_ransac; RANSAC scoring {Hs} x {RS_N}")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_cfg(wl, args.gpus, args.frames or wl["frames"]),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample,
                         "ransac_hyp_pts_per_s": rs},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_reference_c5(args, chk, gen, kind, threads):
    """C5 on the host: `threads` independent sequences, one KLTTracker each (one per host thread), 4 frames per step."""
    from concurrent.futures import ThreadPoolExecutor
    NF = 4
    seqs = [gen.synth_frames(SEED0 + q, 0, NF, C5["W"], C5["H"], threads=1) for q in range(threads)]

    def one(q):
        tr = chk.tracker(max_tracks=C5["corners"], min_tracks=C5["min_tracks"])
        n = 0
        for t in range(NF):
            n += len(tr.tracks()[1]) if t else 0  # tracks entering the step (the first step only resets)
            tr.step(seqs[q][t])
        return n
    times, tracks = [], 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=threads) as ex:
            tracks = sum(ex.map(one, range(threads)))
        if it >= args.warmup:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(times)) if times else float("nan")
    val = tracks / (ms * 1e-3) if times else 0.0
    sample = f"{threads} sequences x {NF} frames per step (one KLTTracker per host thread), {tracks} feature-tracks"
    emit({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": {"workload": f"C5: independent {C5['W']}x{C5['H']} sequences, tracker mode ({C5['corners']} tracks, replenish below {C5['min_tracks']})"},
          "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


# ---------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """Route everything libraries print on fd 1 (e.g. NCCL's version banner) to stderr; the JSON line alone goes to
    the real stdout through emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------------------------
class Unit:
    """One rank's share of a workload: its frames (resident), the pairs object with the RANSAC stage on, host buffers."""

    def __init__(self, ctx, wl, nframes_total, rank, world):
        import sfmgpu
        self.ctx, self.wl, self.rank, self.world = ctx, wl, rank, world
        self.W, self.H, self.cap = wl["W"], wl["H"], wl["corners"]
        self.P_total = nframes_total - 1
        self.p0, self.p1 = shard_range(self.P_total, world, rank)
        self.npairs = self.p1 - self.p0
        self.nfr = self.npairs + 1 if self.npairs > 0 else 0
        self.cfg = sfmgpu.lkcfg(max_tracks=self.cap, pyr_levels=LEVELS)
        self.frames = ctx.frames(self.W, self.H, max(self.nfr, 2), LEVELS)
        self.pairs = ctx.pairs(max(self.npairs, 1), self.cap)
        self.pairs.set_ransac(temple_K(), **RANSAC)
        if self.nfr:
            self.frames.synth(0, self.nfr, SEED0, self.p0)  # this rank's frames of THE sequence: time indices p0 .. p1
        ctx.sync()

    def step_resident(self):
        self.frames.build_pyramid(0, self.nfr)
        self.pairs.run(self.frames, 0, self.npairs, self.cfg)

    def host_buffers(self, with_outputs):
        ctx, P, cap = self.ctx, max(self.npairs, 1), self.cap
        self.host = ctx.pinned_empty((max(self.nfr, 1), self.H, self.W), np.uint8)
        for j in range(self.nfr):  # the device generator is the numpy generator's twin (tests): fill the pinned frames from it
            self.host[j] = self.frames.download(j, 0)
        self.out = None
        if with_outputs:
            self.out = dict(li=ctx.pinned_empty((P, cap, 2), np.float64), lj=ctx.pinned_empty((P, cap, 2), np.float64),
                            nk=ctx.pinned_empty((P,), np.int32), nc=ctx.pinned_empty((P,), np.int32),
                            status=ctx.pinned_empty((P,), np.int32), best_n=ctx.pinned_empty((P,), np.int32),
                            inliers=ctx.pinned_empty((P, cap), np.int32), R=ctx.pinned_empty((P, 9), np.float64),
                            t=ctx.pinned_empty((P, 3), np.float64))
            o = self.out
            self.pairs.ransac_host_outputs(o["status"], o["best_n"], o["inliers"], o["R"], o["t"])
        else:
            self.pairs.ransac_host_outputs()

    def step_host(self, chunk=0):
        o = self.out
        if o is not None:
            self.pairs.run_host(self.frames, self.host[:self.nfr], self.cfg, o["li"], o["lj"], o["nk"], o["nc"], chunk=chunk)
        else:
            self.pairs.run_host(self.frames, self.host[:self.nfr], self.cfg, None, None, None, None, chunk=chunk)

    def close(self):
        self.ctx.sync()
        self.pairs.close()
        self.frames.close()
        for a in [getattr(self, "host", None)] + list((getattr(self, "out", None) or {}).values()):
            if a is not None:
                self.ctx.pinned_free(a)
        self.host = self.out = None


# per-pair layout of a rank's results on the wire: li and the inlier indices are integer-valued and < 32768 -> int16
WIRE = [("li", np.int16, lambda cap: (cap, 2)), ("lj", np.float64, lambda cap: (cap, 2)), ("nk", np.int32, lambda cap: ()),
        ("nc", np.int32, lambda cap: ()), ("status", np.int32, lambda cap: ()), ("best", np.int32, lambda cap: (2,)),
        ("inliers", np.int16, lambda cap: (cap,)), ("R", np.float64, lambda cap: (9,)), ("t", np.float64, lambda cap: (3,))]


def wire_layout(n, cap):
    """[(key, dtype, shape, byte offset)] and the total bytes of one rank's block of n pairs (arrays 8-byte aligned)."""
    out, off = [], 0
    for key, dt, shp in WIRE:
        shape = (n,) + shp(cap)
        out.append((key, dt, shape, off))
        off += (int(np.prod(shape)) * np.dtype(dt).itemsize + 7) // 8 * 8
    return out, off


def gather_to_rank0(unit, torch, dist, shards, hbuf, parts):
    """N > 1: every rank packs its device-resident results into ONE byte block (li and inlier indices as int16) and sends it
    to rank 0 over NCCL (point to point); rank 0 reads each rank's block back to pinned host memory on a side stream while
    the next block arrives."""
    rank, world, n, cap = unit.rank, unit.world, unit.npairs, unit.cap
    v_li, v_lj, v_nk, v_nc = unit.pairs.torch_views(max(n, 1))
    v_st, v_best, v_inl, v_R, v_t = unit.pairs.ransac_torch_views(max(n, 1))
    t_a = time.perf_counter()
    src = dict(li=v_li[:n].to(torch.int16), lj=v_lj[:n], nk=v_nk[:n], nc=v_nc[:n], status=v_st[:n], best=v_best[:n],
               inliers=v_inl[:n].to(torch.int16), R=v_R[:n], t=v_t[:n])
    lay, total = wire_layout(n, cap)
    block = hbuf["send"]
    for key, dt, shape, off in lay:
        nb = int(np.prod(shape)) * np.dtype(dt).itemsize
        block[off:off + nb].copy_(src[key].contiguous().view(torch.uint8).reshape(-1))
    if rank != 0:
        if n > 0:
            dist.send(block[:total], 0)
        torch.cuda.synchronize()
        return
    side = hbuf["stream"]
    for r in range(world):
        a, b = shards[r]
        if b <= a:
            continue
        got = block[:total] if r == 0 else hbuf["dev"][r]
        if r != 0:
            dist.recv(got, r)
        ev = torch.cuda.Event()
        ev.record()
        side.wait_event(ev)
        with torch.cuda.stream(side):
            hbuf["host"][r].copy_(got, non_blocking=True)
    torch.cuda.synchronize()
    parts["gather_and_d2h_ms"] = (time.perf_counter() - t_a) * 1e3


def decode_gathered(hbuf, shards, P, cap):
    """Rank 0: the per-rank byte blocks -> arrays over the whole sequence (outside the timed region: numpy views + one copy)."""
    out = {key: np.zeros((P,) + shp(cap), dt) for key, dt, shp in WIRE}
    for r, (a, b) in enumerate(shards):
        if b <= a:
            continue
        raw = hbuf["host"][r].numpy()
        lay, _ = wire_layout(b - a, cap)
        for key, dt, shape, off in lay:
            nb = int(np.prod(shape)) * np.dtype(dt).itemsize
            out[key][a:b] = raw[off:off + nb].view(dt).reshape(shape)
    return out


DUMP_PAIRS = 128  # pairs whose full lists are dumped: 128 x 8000 corners x (li, lj, inliers) = 40 MB as float64


def dump_outputs(unit, torch, out_dir):
    """What the resident step hands its caller, as DIR/<name>.npy (float64; integers are exact).  Per pair of the sequence:
    n_corners, n_kept, status (0 skipped, 1 no pose, 2 pose), best_h, best_n, R [9], t [3].  For a fixed seeded sample of
    DUMP_PAIRS pairs (pairs.npy): li, lj [cap, 2] and inliers [cap].  Entries the library leaves undefined are zeroed
    (li / lj past n_kept; R, t when status != 2) or -1 (inliers past best_n, or when status != 2)."""
    P = unit.npairs
    v_li, v_lj, v_nk, v_nc = unit.pairs.torch_views(P)
    v_st, v_best, v_inl, v_R, v_t = unit.pairs.ransac_torch_views(P)
    unit.ctx.sync()
    sample = np.sort(np.random.default_rng(SEED0).choice(P, min(P, DUMP_PAIRS), replace=False))
    sel = torch.as_tensor(sample, device=v_li.device)
    nk, st, best = v_nk.cpu().numpy(), v_st.cpu().numpy(), v_best.cpu().numpy()
    ok = st == 2
    out = {"n_corners": v_nc.cpu().numpy(), "n_kept": nk, "status": st, "best_h": best[:, 0], "best_n": best[:, 1],
           "R": np.where(ok[:, None], v_R.cpu().numpy(), 0.0), "t": np.where(ok[:, None], v_t.cpu().numpy(), 0.0), "pairs": sample}
    col = np.arange(unit.cap)
    valid = col[None, :] < nk[sample, None]
    out["li"] = np.where(valid[..., None], v_li[sel].cpu().numpy(), 0.0)
    out["lj"] = np.where(valid[..., None], v_lj[sel].cpu().numpy(), 0.0)
    out["inliers"] = np.where(ok[sample, None] & (col[None, :] < best[sample, 1:2]), v_inl[sel].cpu().numpy(), -1)
    nbytes = sum(a.size * 8 for a in out.values())
    if nbytes > 64 << 20:
        raise ValueError(f"dump of {nbytes} bytes exceeds 64 MB: nothing written")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, np.float64))
    log(f"dumped {len(out)} arrays ({nbytes / 1e6:.1f} MB) of the last timed step to {out_dir}")


def parity_check(chk, gen, wl, sample_pairs, frames_of, got, threads):
    """Reference (chk) on the sampled pairs vs the GPU results `got` (dict of arrays indexed by global pair).  Returns the
    parity_in_bench object."""
    from concurrent.futures import ThreadPoolExecutor
    K = temple_K()

    def one(p):
        fr = frames_of(p)
        _, d = chk.two_view_mt(fr, wl["corners"], 1, K=K, rs_iters=RANSAC["iters"], rs_thr=RANSAC["thr"],
                               rs_min_inliers=RANSAC["min_inliers"], min_points=RANSAC["min_points"])
        return p, d
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=max(1, min(threads, len(sample_pairs)))) as ex:
        res = list(ex.map(one, sample_pairs))
    dt = time.perf_counter() - t0
    ok, worst_lj, worst_R, fails, tracks = True, 0.0, 0.0, [], 0
    for p, d in res:
        nk, nc = int(d["n_kept"][0]), int(d["n_corners"][0])
        tracks += nc
        c = {"n_corners": int(got["nc"][p]) == nc, "n_kept": int(got["nk"][p]) == nk}
        if c["n_kept"]:
            c["li"] = bool(np.array_equal(np.asarray(got["li"][p][:nk], np.float64), d["li"][0, :nk]))
            dev = float(np.abs(got["lj"][p][:nk] - d["lj"][0, :nk]).max()) if nk else 0.0
            worst_lj = max(worst_lj, dev)
            c["lj"] = dev <= KLT_TOL
            c["ransac_status"] = int(got["status"][p]) == int(d["status"][0])
            if c["ransac_status"] and int(d["status"][0]) == 2:
                ni = int(d["n_inl"][0])
                c["ransac_best_n"] = int(got["best_n"][p]) == ni
                c["ransac_inliers"] = c["ransac_best_n"] and bool(np.array_equal(np.asarray(got["inliers"][p][:ni], np.int32), d["inliers"][0, :ni]))
                devR = float(max(np.abs(got["R"][p] - d["R"][0]).max(), np.abs(got["t"][p] - d["t"][0]).max()))
                worst_R = max(worst_R, devR)
                c["pose"] = devR <= POSE_TOL
        if not all(c.values()):
            ok = False
            fails.append({"pair": int(p), "failed": [k for k, v in c.items() if not v]})
    return {"ok": ok, "pairs_checked": [int(p) for p in sample_pairs], "max_lj_dev_px": worst_lj, "lj_tolerance_px": KLT_TOL,
            "max_pose_dev": worst_R, "pose_tolerance": POSE_TOL,
            "pose_note": "R, t come from the device solver's winning hypothesis (equal to the reference's to ~1e-9) through the device "
                         "pose tail; the synthetic sequence has a sub-pixel baseline, so E -> (R, t) is ill-conditioned and amplifies that",
            "bit_exact": ["n_corners", "n_kept", "li", "ransac_status", "ransac_best_n", "ransac_inliers"], "failures": fails,
            "checker": chk.kind}, tracks, dt


def measure_workload(args, ctx, wl, nframes_total, rank, local, world, torch, dist, full):
    """Resident value, stage times, e2e, parity for one workload.  full = the bench line's main workload (clock sampling,
    cpu_baseline); otherwise the shorter side measurement."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    steps = args.steps if full else max(1, min(args.steps, 5))
    warm = args.warmup if full else max(1, min(args.warmup, 2))
    unit = Unit(ctx, wl, nframes_total, rank, world)
    shards = [shard_range(unit.P_total, world, r) for r in range(world)]
    # ---- value: frames resident in HBM ---------------------------------------------------------------------------
    for _ in range(warm):
        unit.step_resident()
    ctx.sync()
    unit.pairs.totals()
    unit.pairs.ransac_early()  # reset the early-stop counter
    barrier()
    sampler = ClockSampler(local) if (full and rank == 0) else None
    if sampler:
        sampler.start()
    l0 = ctx.launches()
    ctx.timer_start()
    for _ in range(steps):
        unit.step_resident()
    ms_total = ctx.timer_stop()
    launches = ctx.launches() - l0
    barrier()
    clocks = sampler.stop() if sampler else None
    n_tracks, n_kept, n_it = unit.pairs.totals()
    early_pairs = unit.pairs.ransac_early()  # pair-steps whose RANSAC scoring stopped at a full count (exact, see DESIGN.md §4)
    if full and args.dump_outputs:
        dump_outputs(unit, torch, args.dump_outputs)  # before the passes below overwrite the results

    # ---- the same step with every hypothesis of every pair solved and scored (early stop off) --------------------------------
    fs_steps = max(1, min(steps, 3))
    ctx.ransac_set_early_stop(False)
    unit.step_resident()
    ctx.sync()
    barrier()
    ctx.timer_start()
    for _ in range(fs_steps):
        unit.step_resident()
    fs_ms = ctx.timer_stop() / fs_steps
    ctx.ransac_set_early_stop(True)
    unit.pairs.totals()
    unit.pairs.ransac_early()
    barrier()

    # ---- per-stage times (separate pass, stages back to back on one stream) ------------------------------------------
    ctx.profile(True)
    ctx.timer_start()
    unit.frames.build_pyramid(0, unit.nfr)
    pyr_ms = ctx.timer_stop()
    unit.pairs.run(unit.frames, 0, unit.npairs, unit.cfg)
    st = ctx.stage_times()
    ctx.profile(False)

    # ---- e2e: host (pinned) frames in, tracks + inlier sets + poses out ---------------------------------------------------
    unit.host_buffers(with_outputs=(world == 1))
    o = unit.out
    h2d = unit.nfr * unit.W * unit.H
    d2h = sum(a.nbytes for a in o.values()) if o else 0
    hbuf, parts = None, {}
    if world > 1:
        P, cap = unit.P_total, unit.cap
        sizes = [wire_layout(b - a, cap)[1] for a, b in shards]
        hbuf = {"send": torch.empty(max(sizes[rank], 8), dtype=torch.uint8, device="cuda")}
        if rank == 0:
            hbuf["host"] = {r: torch.empty(max(sizes[r], 8), dtype=torch.uint8, pin_memory=True) for r in range(world)}
            hbuf["dev"] = {r: torch.empty(max(sizes[r], 8), dtype=torch.uint8, device="cuda") for r in range(1, world)}
            hbuf["stream"] = torch.cuda.Stream()
            d2h = sum(sizes)

    def step_e2e():
        if world == 1:
            unit.step_host(chunk=args.chunk)
            return
        t_a = time.perf_counter()
        unit.step_host(chunk=args.chunk)
        ctx.sync()  # results are written on the library's streams; NCCL runs on torch's
        parts["stream_call_ms"] = (time.perf_counter() - t_a) * 1e3
        gather_to_rank0(unit, torch, dist, shards, hbuf, parts)

    # the PCIe floor: every rank uploads its frames at the same time, nothing else (max over ranks below)
    unit.frames.upload_ptr(0, unit.nfr, unit.host.ctypes.data)
    barrier()
    t0 = time.perf_counter()
    unit.frames.upload_ptr(0, unit.nfr, unit.host.ctypes.data)
    ctx.sync()
    h2d_floor_ms = (time.perf_counter() - t0) * 1e3
    barrier()

    e2e_steps = max(1, min(steps, 3))
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    ctx.timer_start()
    for _ in range(e2e_steps):
        step_e2e()
    e2e_ms_dev = ctx.timer_stop()
    barrier()
    e2e_wall = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(e2e_ms_dev, e2e_wall) / e2e_steps

    # results of the e2e step, indexed by global pair, on rank 0
    got = None
    if world == 1:
        assert int(o["nc"].sum()) == n_tracks and int(o["nk"].sum()) == n_kept, "e2e results differ from the resident run"
        got = dict(o)
    elif rank == 0:
        h = decode_gathered(hbuf, shards, unit.P_total, unit.cap)
        got = dict(li=h["li"], lj=h["lj"], nk=h["nk"], nc=h["nc"], status=h["status"], best_n=h["best"][:, 1], inliers=h["inliers"],
                   R=h["R"], t=h["t"])
        a, b = shards[0]
        assert int(got["nc"][a:b].sum()) == n_tracks and int(got["nk"][a:b].sum()) == n_kept, "gathered results differ from the resident run"

    # ---- parity inside the bench + CPU baseline (rank 0) ---------------------------------------------------------------------
    parity, cpu = None, None
    if rank == 0 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle
        chk, kind = oracle.best()
        gen = oracle.port()
        threads = host_threads()
        if world == 1:
            sample = list(range(min(threads, unit.P_total)))
            frames_of = lambda p: np.ascontiguousarray(unit.host[p:p + 2])
        else:
            # the first pair of every rank's block (offsets and halo frames of the sharding), then the pairs after them
            sample = []
            for k in range(max(1, threads // world)):
                sample += [a + k for a, b in shards if a + k < b]
            sample = sorted(set(sample))[:threads]
            frames_of = lambda p: gen.synth_frames(SEED0, p, 2, unit.W, unit.H, threads=1)
        parity, ptracks, pdt = parity_check(chk, gen, wl, sample, frames_of, got, threads)
        if full and world == 1:
            xi, xj = c4_points(RS_N)
            Hs = 64 * threads
            E = np.ascontiguousarray(np.tile(chk.ransac_hypotheses(xi, xj, 64)[0], (threads, 1)))
            t1 = time.perf_counter()
            chk.ransac_score_mt(xi, xj, E, 1e-3, threads)
            rs = Hs * RS_N / (time.perf_counter() - t1)
            t2 = time.perf_counter()
            one_tracks, _ = chk.two_view_mt(np.ascontiguousarray(unit.host[:2]), wl["corners"], 1, K=temple_K(), rs_iters=RANSAC["iters"],
                                            rs_thr=RANSAC["thr"], rs_min_inliers=RANSAC["min_inliers"], min_points=RANSAC["min_points"],
                                            detail=False)
            one_core = one_tracks / (time.perf_counter() - t2)
            cpu = {"value": ptracks / pdt, "unit": UNIT, "cores": min(threads, len(sample)), "kind": kind, "one_core_value": one_core,
                   "sample": f"first {len(sample)} pairs of the same sequence, one per host thread, front end + find_E_ransac "
                             f"({ptracks} feature-tracks in {pdt:.2f} s wall); the same run is the parity_in_bench check",
                   "ransac_hyp_pts_per_s": rs}

    # ---- reduce over ranks ------------------------------------------------------------------------------------------------
    ms_step = ms_total / steps
    vals = torch.tensor([ms_step, e2e_ms, pyr_ms, st["klt"], st["corner_score"], st["corner_select"], st["ransac"], st["compact"], h2d_floor_ms,
                         fs_ms], device="cuda", dtype=torch.float64)
    work = torch.tensor([n_tracks, n_kept, n_it, launches, h2d, early_pairs], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(work, op=dist.ReduceOp.SUM)
    ms_step, e2e_ms, pyr_ms, klt_ms, cs_ms, sel_ms, rs_ms, cp_ms, h2d_floor_ms, fs_ms = [float(v) for v in vals.tolist()]
    tracks_all, kept_all, it_all, launches_all, h2d_all, early_all = [int(v) for v in work.tolist()]
    unit.close()
    res = dict(ms_step=ms_step, e2e_ms=e2e_ms, e2e_steps=e2e_steps, pyr_ms=pyr_ms, klt_ms=klt_ms, cs_ms=cs_ms, sel_ms=sel_ms, rs_ms=rs_ms,
               cp_ms=cp_ms, h2d_floor_ms=h2d_floor_ms, tracks=tracks_all, kept=kept_all, iters=it_all, launches=launches_all, h2d=h2d_all,
               d2h=d2h, parity=parity, cpu=cpu, clocks=clocks, parts=parts, steps=steps, warmup=warm, nframes=nframes_total,
               pairs_rank0=unit.npairs, frames_rank0=unit.nfr, fs_ms=fs_ms, fs_steps=fs_steps, early_pairs=early_all,
               pair_steps=unit.P_total * steps)
    return res


C5 = dict(name="C5", W=1920, H=1080, sequences=64, frames=64, corners=2000, min_tracks=818)


def measure_c5(args, ctx, rank, local, world, torch, dist, steps, warm, frames_per_seq, check=True):
    """BASELINE.json configs[4]: a batch of 64 independent 1080p sequences across the GPUs of the box, TRACKER mode
    (KLTTracker::step semantics per sequence, cpp/src/templering_sfm.cpp:340-391: tracks chain from frame to frame, replenish
    below min_tracks).  Rank g owns sequences [g*64/N, (g+1)*64/N) and advances them in lock step (sfmgpu_multitracker: one
    batched launch per stage and step; the next frames travel while the current ones compute).  One bench step = all frames
    of all sequences.  value: source frames resident in HBM; e2e: source frames in pinned host memory."""
    import sfmgpu
    W, H, T = C5["W"], C5["H"], frames_per_seq
    s0, s1 = shard_range(C5["sequences"], world, rank)
    S = s1 - s0
    cfg = sfmgpu.lkcfg(max_tracks=C5["corners"], min_tracks=C5["min_tracks"], pyr_levels=LEVELS)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    res = dict(S=S, T=T, tracks=0, ms=float("nan"), e2e_ms=float("nan"), parity=None, launches=0, h2d=0)
    if S > 0:
        store = ctx.frames(W, H, T * S, 1)  # frame t of sequence s at index t*S + s: one lock-step's frames are contiguous
        for t in range(T):
            for q in range(S):
                store.synth(t * S + q, 1, SEED0 + s0 + q, t)
        base, pitch, fstride = store.device_ptr(0)
        assert pitch == W and fstride == W * H, "1080p rows are 16-byte multiples: the store is dense"
        host = ctx.pinned_empty((T, S, H, W), np.uint8)
        for k in range(T * S):
            host.reshape(T * S, H, W)[k] = store.download(k, 0)
        mt = ctx.multitracker(S, W, H, cfg)
        step_bytes = S * W * H

        def one_pass(src):
            mt.reset()
            for t in range(T):
                nxt = src + (t + 1) * step_bytes if t + 1 < T else None
                mt.step_ptr(src if t == 0 else None, nxt)
            return mt.totals()[0]

        for _ in range(warm):
            one_pass(base)
    barrier()
    if S > 0:
        l0 = ctx.launches()
        t0 = time.perf_counter()
        ctx.timer_start()
        for _ in range(steps):
            tracks = one_pass(base)
        ms_dev = ctx.timer_stop()
        res["ms"] = max(ms_dev, (time.perf_counter() - t0) * 1e3) / steps  # the lock-step loop synchronises every step: wall == device
        res["launches"] = ctx.launches() - l0
        res["tracks"] = tracks
    barrier()
    if S > 0:
        one_pass(host.ctypes.data)
    barrier()
    if S > 0:
        e2e_steps = max(1, min(steps, 3))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            one_pass(host.ctypes.data)
        ctx.sync()
        res["e2e_ms"] = (time.perf_counter() - t0) * 1e3 / e2e_steps
        res["h2d"] = T * step_bytes
    barrier()
    # parity: the first and the last sequence of rank 0 against the reference tracker on the first frames (ids bit-exact,
    # positions within the KLT tolerance, the track list after every step)
    if check and rank == 0 and S > 0 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle
        from concurrent.futures import ThreadPoolExecutor
        chk, kind = oracle.best()
        nchk = min(T, 8)
        seqs = sorted({0, S - 1})
        mt.reset()
        got = []
        for t in range(nchk):
            out = mt.step(host[t])
            got.append([(out[q], mt.tracks(q)) for q in seqs])

        def ref_seq(q):
            tr = chk.tracker(max_tracks=C5["corners"], min_tracks=C5["min_tracks"])
            outs = []
            for t in range(nchk):
                o = tr.step(host[t, q])
                outs.append((o, tr.tracks()))
            return outs
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=len(seqs)) as ex:
            want = list(ex.map(ref_seq, seqs))
        ok, worst, nsteps = True, 0.0, 0
        for k, q in enumerate(seqs):
            for t in range(nchk):
                (gp, gc, gi), (gxy, gids) = got[t][k]
                (wp, wc, wi), (wxy, wids) = want[k][t]
                same = len(gi) == len(wi) and np.array_equal(gi, wi) and np.array_equal(gids, wids)
                if same and len(gi):
                    dev = max(float(np.abs(gp - wp).max()), float(np.abs(gc - wc).max()), float(np.abs(gxy - wxy).max()))
                    worst = max(worst, dev)
                    same = dev <= KLT_TOL
                ok = ok and same
                nsteps += 1
        res["parity"] = {"ok": ok, "sequences_checked": [int(s0 + q) for q in seqs], "steps_each": nchk, "max_pos_dev_px": worst,
                         "tolerance_px": KLT_TOL, "bit_exact": ["survivor ids", "track-list ids"], "checker": kind,
                         "reference_s": time.perf_counter() - t0}
    if S > 0:
        mt.close()
        store.close()
        ctx.pinned_free(host)
    vals = torch.tensor([res["ms"] if S else 0.0, res["e2e_ms"] if S else 0.0], device="cuda", dtype=torch.float64)
    work = torch.tensor([res["tracks"], res["launches"], res["h2d"]], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(work, op=dist.ReduceOp.SUM)
    res["ms"], res["e2e_ms"] = [float(v) for v in vals.tolist()]
    res["tracks"], res["launches"], res["h2d"] = [int(v) for v in work.tolist()]
    return res


def c5_block(r, world, steps, warm):
    return {"config": f"C5: {C5['sequences']} independent synthetic {C5['W']}x{C5['H']} sequences x {r['T']} frames, tracker mode "
                      f"(KLTTracker::step per sequence: {C5['corners']} tracks, replenish below {C5['min_tracks']}), "
                      f"{C5['sequences'] // world if C5['sequences'] % world == 0 else str(C5['sequences']) + '/' + str(world)} sequences per GPU in lock step",
            "value": r["tracks"] / (r["ms"] * 1e-3), "unit": UNIT, "ms_per_step": r["ms"], "steps": steps, "warmup": warm,
            "lockstep_steps_per_s": C5["sequences"] * r["T"] / (r["ms"] * 1e-3),
            "e2e_value": r["tracks"] / (r["e2e_ms"] * 1e-3), "e2e_ms_per_step": r["e2e_ms"], "h2d_bytes_per_step": r["h2d"],
            "feature_tracks_per_step": r["tracks"], "gpu_launches": r["launches"], "scaling": "strong",
            "parity_in_bench": r["parity"]["ok"] if r["parity"] else None, "parity_detail": r["parity"]}


def stage_block(wl, r, world, hbm_peak):
    per_rank_tracks = r["tracks"] / world
    nfr, W, H = r["frames_rank0"], wl["W"], wl["H"]
    pyr_bytes = nfr * W * H * sum(0.25 ** l for l in range(LEVELS))
    cs_bytes = r["pairs_rank0"] * W * H
    klt_gbs = B_KLT * per_rank_tracks / (r["klt_ms"] * 1e-3) / 1e9
    return {
        "stages_ms": {"pyramid": r["pyr_ms"], "corner_score": r["cs_ms"], "corner_select": r["sel_ms"], "klt": r["klt_ms"],
                      "compact": r["cp_ms"], "ransac": r["rs_ms"]},
        "ransac_early_stop": {
            "pairs_stopped_fraction": r["early_pairs"] / max(r["pair_steps"], 1),
            "full_scoring": {"value": r["tracks"] / (r["fs_ms"] * 1e-3), "unit": UNIT, "ms_per_step": r["fs_ms"], "steps": r["fs_steps"]},
            "note": "exact: the scoring loop keeps the FIRST hypothesis with the largest count (:673) and a count cannot exceed the number of "
                    "points, so a pair whose first 128 hypotheses contain one that explains all of its points is not solved / scored "
                    "further (same winner, inlier list, pose; DESIGN.md §4).  On this synthetic sequence - as on any pair whose "
                    "correspondences all lie within the reference's 2e-3 Sampson threshold (tens of pixels) of an early hypothesis - that is "
                    "every pair.  full_scoring = the same resident step with the stop off (all iters hypotheses of every pair solved and "
                    "scored, as the reference does); value / ms_per_step / stages_ms of the line are with the stop on (the library's default)"},
        "stage_rooflines": {
            "pyramid": {"bound": "hbm", "achieved": pyr_bytes / (r["pyr_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": pyr_bytes / (r["pyr_ms"] * 1e-3) / 1e9 / hbm_peak},
            "corner_score": {"bound": "hbm", "achieved": cs_bytes / (r["cs_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": cs_bytes / (r["cs_ms"] * 1e-3) / 1e9 / hbm_peak, "mpx_per_s": cs_bytes / (r["cs_ms"] * 1e-3) / 1e6},
            "klt": {"bound": "hbm", "achieved": klt_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": klt_gbs / hbm_peak},
        },
    }


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c5"],
                    help="c3 (default): 4K x 2000 frames, 8000 corners, pair-sharded; c2: 1080p x 1000 frames, 2000 corners; "
                         "c5: 64 independent 1080p sequences in tracker mode (attached to the default line as 'c5')")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 side measurement of the default line")
    ap.add_argument("--no-shim", action="store_true", help="skip the C++ shim timings (find_E_ransac, loop-closure block): profiling runs")
    ap.add_argument("--frames", type=int, default=0, help="frames of the sequence (default: the workload's own length)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (cpu_baseline, parity_in_bench)")
    ap.add_argument("--no-c2", action="store_true", help="skip the C2 side measurement of the default line")
    ap.add_argument("--pipe", type=int, default=-1, help="pairs per sub-chunk of the stage pipeline (-1: library default, 0: off)")
    ap.add_argument("--klt-mode", type=int, default=0, help="sfmgpu_klt_set_mode value (A/B timing of kernel variants)")
    ap.add_argument("--chunk", type=int, default=0, help="frames per chunk of the streaming e2e call (0: library default, about 100 frames)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the results of the last timed step to DIR/<name>.npy (float64, at most 64 MB; c3 / c2, one process), "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "c5" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs covers the two-view workloads (c3, c2) of --impl ours in one process")
    args.warmup = max(args.warmup, 0)
    wl = WORKLOADS["c3" if args.workload == "c5" else args.workload]
    nframes_total = args.frames or wl["frames"]

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, wl, rank)
        return

    import torch
    import torch.distributed as dist
    import sfmgpu

    torch.cuda.set_device(local)
    near_cpus = bind_near_gpu(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = sfmgpu.Context(local)  # raises without the CUDA library / device: there is no CPU fallback
    if args.pipe >= 0:
        ctx.pipeline_set(args.pipe)
    if args.klt_mode:
        ctx.klt_set_mode(args.klt_mode)

    if args.workload == "c5":
        run_c5_line(args, ctx, rank, local, world, torch, dist, near_cpus)
        return
    r = measure_workload(args, ctx, wl, nframes_total, rank, local, world, torch, dist, full=True)
    c5 = None
    if args.workload == "c3" and not args.no_c5 and not args.frames:
        c5 = measure_c5(args, ctx, rank, local, world, torch, dist, max(1, min(args.steps, 3)), 1, C5["frames"], check=(world == 1))
    c2 = None
    if args.workload == "c3" and world == 1 and not args.no_c2 and not args.frames:
        c2 = measure_workload(args, ctx, WORKLOADS["c2"], WORKLOADS["c2"]["frames"], rank, local, world, torch, dist, full=False)
    fp64_peak = ctx.fp64_peak()

    # ---- RANSAC half of the metric (C4), rank-local: the seeded sampler's octets through the device solver, then scoring ------
    xi, xj = c4_points(RS_N)
    idx8 = ctx.ransac_sample(RS_N, RS_H * 8).reshape(RS_H, 8)
    solver = {}
    for mode in (3, 0):  # 3: screening solver (what the batched stage counts with), 0: Jacobi emulation for every octet
        ctx.solver_set_mode(mode)
        ctx.ransac_hypotheses(xi, xj, idx8, fetch=False)
        ctx.sync()
        ctx.timer_start()
        ctx.ransac_hypotheses(xi, xj, idx8, fetch=False)
        solver[mode] = ctx.timer_stop()
    ctx.solver_set_mode(1)
    solver_ms, screen_ms = solver[0], solver[3]  # the scoring rate below is measured on the emulation's hypotheses
    for _ in range(3):
        ctx.ransac_score_resident(1e-3, fetch=False)
    ctx.sync()
    ctx.timer_start()
    RS_REP = 10
    for _ in range(RS_REP):
        ctx.ransac_score_resident(1e-3, fetch=False)
    rs_ms = ctx.timer_stop() / RS_REP
    bh, bn = ctx.ransac_score_resident(1e-3)

    # ---- the reference's own two-view entry point through the C++ shim (TempleRing-sized call, sfm.cpp:1739) ---------------------
    find_e = None
    if rank == 0 and not args.no_shim:
        try:
            import ctypes as C
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import shimlib
            from conftest import TEMPLE_K, two_view_scene
            shim = shimlib.load()
            pi, pj = two_view_scene(2200, seed=2200)
            Kf = np.ascontiguousarray(TEMPLE_K.reshape(9))
            Rr, tt, il, kk = np.zeros(9), np.zeros(3), np.zeros(2200, np.int32), C.c_int(0)
            find_e = {"iters": 2500, "points": 2200}
            for name, flag in (("host_solver_ms", 0), ("device_solver_ms", 1)):
                shim.shim_set_device_solver(flag)
                shim.shim_find_E_ransac(Kf, pi, pj, 2200, 2500, 1e-3, 60, Rr, tt, il, C.byref(kk))
                t0 = time.perf_counter()
                for _ in range(3):
                    shim.shim_find_E_ransac(Kf, pi, pj, 2200, 2500, 1e-3, 60, Rr, tt, il, C.byref(kk))
                find_e[name] = (time.perf_counter() - t0) / 3 * 1e3
                find_e[name.replace("_ms", "_inliers")] = int(kk.value)
            shim.shim_set_device_solver(0)
            # the loop-closure block (:1841-1852) through the shim on a TempleRing-sized pair, as the reference writes it
            # (track_one_public per corner: one launch + sync each, 2 x 1200 per loop closure) and with the batched call
            from sfmgpu import synth
            f0, f1 = synth.frame(SEED0, 0, 640, 480), synth.frame(SEED0, 1, 640, 480)
            lli, llj, nn = np.zeros((1200, 2)), np.zeros((1200, 2)), C.c_int(0)
            find_e["loop_closure_block"] = {"image": "640x480", "max_corners": 1200}
            for name, batched in (("per_point_ms", 0), ("batched_ms", 1)):
                shimlib.ck(shim, shim.shim_pair_frontend(f0, f1, 640, 480, 1200, 0.01, 8, 3, 5, 10, 1.0, batched, lli, llj, C.byref(nn)))
                t0 = time.perf_counter()
                kept = shimlib.ck(shim, shim.shim_pair_frontend(f0, f1, 640, 480, 1200, 0.01, 8, 3, 5, 10, 1.0, batched, lli, llj, C.byref(nn)))
                find_e["loop_closure_block"][name] = (time.perf_counter() - t0) * 1e3
                find_e["loop_closure_block"]["corners"] = int(nn.value)
                find_e["loop_closure_block"]["kept"] = int(kept)
        except Exception as ex:  # the shim is optional for the bench line
            find_e = {"error": str(ex)[:200]}

    rs_t = torch.tensor([rs_ms, solver_ms, screen_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(rs_t, op=dist.ReduceOp.MAX)
    rs_ms, solver_ms, screen_ms = [float(v) for v in rs_t.tolist()]

    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        prof = profile_metrics()
        value = r["tracks"] / (r["ms_step"] * 1e-3)
        e2e_val = r["tracks"] / (r["e2e_ms"] * 1e-3)
        blk = stage_block(wl, r, world, hbm_peak)
        stage = blk["stages_ms"]
        dominant = max(("klt", "corner_score", "corner_select", "ransac"), key=lambda k: stage[k])
        kq = prof.get("klt_quad_kernel", {})
        traffic = (kq.get("dram_read_bytes", 0) + kq.get("dram_write_bytes", 0)) or None
        klt_gbs = blk["stage_rooflines"]["klt"]["achieved"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": r["steps"], "warmup": r["warmup"],
            "ms_per_step": r["ms_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_cfg(wl, world, nframes_total),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": int(r["d2h"]),
                    "gather": "none (1 GPU)" if world == 1 else f"NCCL point-to-point, one packed block per rank to rank 0 ({world} ranks), li and inlier indices as int16; "
                              "rank 0 reads each block back while the next arrives",
                    "cpus_bound_near_gpu": near_cpus, "rank0_parts_ms": r["parts"] or None, "ms_per_step": r["e2e_ms"], "steps": r["e2e_steps"],
                    "h2d_floor_ms": r["h2d_floor_ms"], "h2d_floor_gb_per_s": r["h2d"] / (r["h2d_floor_ms"] * 1e-3) / 1e9,
                    "floor_over_e2e": r["h2d_floor_ms"] / r["e2e_ms"],
                    "note": "h2d_floor_ms = all ranks upload their frames at the same time and do nothing else (max over ranks): the "
                            "PCIe / host-memory floor of the end-to-end step at this N"},
            "parity_in_bench": r["parity"]["ok"] if r["parity"] else None,
            "parity_detail": r["parity"],
            "gpu_launches": r["launches"],
            "clocks": r["clocks"],
            "roofline": {"bound": "hbm", "kernel": "klt_quad_kernel (+ klt_lane_kernel<...,masked> / klt_kernel<5,true> on border features)",
                         "achieved": klt_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": klt_gbs / hbm_peak, "traffic": traffic,
                         "traffic_source": f"dram__bytes_read+write of one klt_quad_kernel launch, ncu --set full ({kq.get('source', 'profiles/')}; static, not re-measured)",
                         "peak_source": peak_src, "dominant_stage_by_time": dominant,
                         "note": "KLT is the largest front-end stage; it is bound by instruction issue (integer-valued FP32 matrix build + FP64 "
                                 "iterations), not HBM (SURVEY.md §8d: ~140 flop/B), so the HBM fraction is a few percent by construction; "
                                 "stage_rooflines has the HBM-bound stages (pyramid, corner score)"},
            "roofline_issue": {"kernel": "klt_quad_kernel", "bound": "instruction issue",
                               "issue_active_frac_static": (kq.get("issue_active_pct") or 0) / 100.0 or None,
                               "fp64_pipe_frac_static": (kq.get("fp64_pipe_pct") or 0) / 100.0 or None,
                               "source": f"{kq.get('source', 'profiles/')} (ncu smsp__issue_active / sm__pipe_fp64_cycles_active: STATIC quote of the committed capture, not measured in this run)",
                               "reference_formulation_tflops": F_KLT_IT * (r["iters"] / world) / (r["klt_ms"] * 1e-3) / 1e12,
                               "fp64_peak_tflops": fp64_peak, "fp64_peak_source": "in-run DFMA micro-benchmark (sfmgpu_fp64_peak)",
                               "flop_per_lk_iteration_reference": F_KLT_IT, "lk_iterations": r["iters"]},
            "stages_ms": blk["stages_ms"], "stage_rooflines": blk["stage_rooflines"], "ransac_early_stop": blk["ransac_early_stop"],
            "kept_fraction": r["kept"] / max(r["tracks"], 1),
            "ransac": {"value": RS_H * RS_N / (rs_ms * 1e-3), "unit": "hyp*pts/s", "ms": rs_ms, "hypotheses": RS_H, "points": RS_N,
                       "solver_ms": solver_ms, "solver_hyp_per_s": RS_H / (solver_ms * 1e-3),
                       "screen_solver_ms": screen_ms, "screen_solver_hyp_per_s": RS_H / (screen_ms * 1e-3),
                       "solver_note": "solver_ms: Jacobi emulation of eight_point_E for every octet; screen_solver_ms: the null vector by Householder QR, "
                                      "which the batched stage counts with (the winner of every pair is re-solved by the emulation)", "best_h": int(bh), "best_inliers": int(bn),
                       "reference_formulation_tflops_over_fp64_peak": F_RS * RS_H * RS_N / (rs_ms * 1e-3) / 1e12 / fp64_peak,
                       "issue_active_frac_static": (prof.get("ransac_count_kernel", {}).get("issue_active_pct") or 0) / 100.0 or None,
                       "hypotheses_source": "device sampler (std::mt19937(12345) + uniform_int_distribution, bit-exact octets) + device 8-point solver on the C4 points",
                       "find_E_ransac": find_e},
        }
        if r["cpu"]:
            line["cpu_baseline"] = r["cpu"]
        if c2:
            b2 = stage_block(WORKLOADS["c2"], c2, world, hbm_peak)
            line["c2"] = {"config": workload_cfg(WORKLOADS["c2"], world, c2["nframes"])["workload"], "value": c2["tracks"] / (c2["ms_step"] * 1e-3),
                          "ms_per_step": c2["ms_step"], "steps": c2["steps"], "warmup": c2["warmup"],
                          "e2e_value": c2["tracks"] / (c2["e2e_ms"] * 1e-3), "e2e_ms_per_step": c2["e2e_ms"], "h2d_floor_ms": c2["h2d_floor_ms"],
                          "parity_in_bench": c2["parity"]["ok"] if c2["parity"] else None, "parity_detail": c2["parity"],
                          "stages_ms": b2["stages_ms"], "stage_rooflines": b2["stage_rooflines"], "ransac_early_stop": b2["ransac_early_stop"],
                          "kept_fraction": c2["kept"] / max(c2["tracks"], 1)}
        if c5:
            line["c5"] = c5_block(c5, world, max(1, min(args.steps, 3)), 1)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_c5_line(args, ctx, rank, local, world, torch, dist, near_cpus):
    """--workload c5 as the bench line itself."""
    T = args.frames or C5["frames"]
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    r = measure_c5(args, ctx, rank, local, world, torch, dist, args.steps, args.warmup, T)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        blk = c5_block(r, world, args.steps, args.warmup)
        hbm_peak, peak_src = measured_peaks()
        klt_gbs = B_KLT * r["tracks"] / world / (r["ms"] * 1e-3) / 1e9
        line = {"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": {"workload": blk["config"], "sequences": C5["sequences"], "frames_per_sequence": T,
                                                "width": C5["W"], "height": C5["H"], "max_tracks": C5["corners"], "min_tracks": C5["min_tracks"],
                                                "sharding": f"whole sequences per rank x{world}, lock step per rank, no collective",
                                                "l2_policy": "every lock-step reads fresh frames (133 MB per 64 sequences): no reuse across steps"},
                "e2e": {"value": blk["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": 4 * C5["sequences"] * T,
                        "ms_per_step": r["e2e_ms"], "cpus_bound_near_gpu": near_cpus,
                        "note": "frames come from pinned host memory, the next lock-step's frames travel while the current one computes; "
                                "survivor counts return every step (the track lists stay on the device until asked for)"},
                "parity_in_bench": blk["parity_in_bench"], "parity_detail": blk["parity_detail"], "gpu_launches": r["launches"], "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "KLT chain of the lock-step tracker", "achieved": klt_gbs, "peak": hbm_peak, "unit": "GB/s",
                             "frac": klt_gbs / hbm_peak, "traffic": None, "peak_source": peak_src,
                             "note": "whole lock-step (upload wait + pyramid + KLT + compaction + replenish) over the KLT algorithmic bytes"},
                "lockstep_steps_per_s": blk["lockstep_steps_per_s"]}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
