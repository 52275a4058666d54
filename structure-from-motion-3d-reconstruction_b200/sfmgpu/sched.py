"""Multi-GPU frame-pair / sequence scheduler (SURVEY.md §8e) - the torch.distributed face, used by bench.py and the
gloo tests.  The C++ drop-in uses the same sharding through the C ABI (include/sfmgpu.h: sfmgpu_sched_*, csrc/sched.cu,
NCCL send / recv); `shard_range` below IS that C function, so both faces agree by construction.

The front end shards with NO data-path collective:
  * pair mode     - the stateless two-view unit (cpp/src/templering_sfm.cpp:1836-1857): pairs (t, t+1) are independent;
                    rank g owns a contiguous block of pairs plus one halo frame (`pair_shard`);
  * sequence mode - whole sequences per rank (a KLTTracker chain cannot be split across frames, :370-371): `shard_range`
                    over the sequences; several sequences per GPU advance in lock step (run_sequences -> sfmgpu_multitracker);
  * segment mode  - contiguous frame segments of one sequence, each restarting the tracker: `segment_shard` spreads G
                    segments of equal length over the sequence and gives each rank a block of them (Pairs.run_segments
                    runs them).  That equals the reference run on each segment separately (track ids restart per
                    segment), NOT the unsegmented run.
The only communication is the gather of results (tracks, survivor counts, inlier sets) to rank 0: an all_gather of
per-rank sizes followed by one padded gather (NCCL has no gatherv).  Works on NCCL (GPU tensors) and gloo (CPU tests).
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_items, world, rank):
    """Contiguous block [start, end) of n_items for `rank`; sizes differ by at most one, lower ranks get the extra.
    Calls sfmgpu_sched_shard (a pure function of the C ABI: no GPU needed)."""
    import sfmgpu
    lib = sfmgpu.load_library()
    a, b = C.c_int(0), C.c_int(0)
    if lib.sfmgpu_sched_shard(int(n_items), int(world), int(rank), C.byref(a), C.byref(b)) != 0:
        raise ValueError(f"shard_range({n_items}, {world}, {rank})")
    return a.value, b.value


def pair_shard(n_frames, world, rank):
    """Pairs [p0, p1) of a sequence of n_frames and the frames [p0, p1] (inclusive halo) the rank must hold."""
    p0, p1 = shard_range(max(n_frames - 1, 0), world, rank)
    return p0, p1, (p0, p1 + 1 if p1 > p0 else p0)


class _RankOf(C.Structure):
    """The head of sfmgpu_sched that the shard functions read (csrc/sched.cu asserts the layout)."""
    _fields_ = [("world", C.c_int), ("rank", C.c_int)]


def segment_shard(n_frames, n_segments, world=1, rank=0):
    """Segment mode: sfmgpu_sched_segment_shard (no GPU needed).  Returns (steps, seg_begin, seg_end, seg_first [n_segments]
    int32, frame_begin, frame_end): this rank runs segments [seg_begin, seg_end) of `steps` steps each, segment j starting on
    frame seg_first[j], and must hold frames [frame_begin, frame_end)."""
    import sfmgpu
    lib = sfmgpu.load_library()
    L, a, b, f0, f1 = (C.c_int(0) for _ in range(5))
    first = np.zeros(max(int(n_segments), 1), np.int32)
    if lib.sfmgpu_sched_segment_shard(C.byref(_RankOf(int(world), int(rank))), int(n_frames), int(n_segments), C.byref(L), C.byref(a),
                                      C.byref(b), first.ctypes.data_as(C.c_void_p), C.byref(f0), C.byref(f1)) != 0:
        raise ValueError(f"segment_shard({n_frames}, {n_segments}, {world}, {rank})")
    return L.value, a.value, b.value, first[:n_segments], f0.value, f1.value


def _dev(t):
    return t.device


def gather_rows(local, dst=0):
    """Gather 2-D tensors with different numbers of rows to `dst`.  Returns the list of per-rank tensors on dst,
    None elsewhere.  One all_gather of row counts + one padded gather."""
    world, rank = dist.get_world_size(), dist.get_rank()
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=_dev(local))
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    cap = max(max(sizes), 1)
    pad = torch.zeros((cap,) + tuple(local.shape[1:]), dtype=local.dtype, device=_dev(local))
    pad[: local.shape[0]] = local
    out = [torch.empty_like(pad) for _ in range(world)] if rank == dst else None
    dist.gather(pad, out, dst=dst)
    if rank != dst:
        return None
    return [o[:s] for o, s in zip(out, sizes)]


def gather_pair_results(n_kept, li, lj, dst=0):
    """Per-rank results of a block of pairs -> rank `dst`.
    n_kept: int32 [P]; li, lj: float64 [P, cap, 2] (first n_kept[p] rows of pair p are valid).
    Returns (n_kept_all [sum P], li_list, lj_list) on dst with pairs in global order, None elsewhere."""
    dev = _dev(n_kept)
    flat_i = torch.cat([li[p, : int(n_kept[p])] for p in range(li.shape[0])]) if li.shape[0] else torch.zeros((0, 2), dtype=li.dtype, device=dev)
    flat_j = torch.cat([lj[p, : int(n_kept[p])] for p in range(lj.shape[0])]) if lj.shape[0] else torch.zeros((0, 2), dtype=lj.dtype, device=dev)
    counts = gather_rows(n_kept.reshape(-1, 1).to(torch.int64), dst)
    gi = gather_rows(flat_i, dst)
    gj = gather_rows(flat_j, dst)
    if dist.get_rank() != dst:
        return None
    counts = torch.cat(counts).reshape(-1)
    fi, fj = torch.cat(gi), torch.cat(gj)
    offs = np.concatenate([[0], np.cumsum(counts.cpu().numpy())])
    li_list = [fi[offs[k]:offs[k + 1]] for k in range(len(counts))]
    lj_list = [fj[offs[k]:offs[k + 1]] for k in range(len(counts))]
    return counts, li_list, lj_list


def run_sequences(sequences, device=0, lkcfg_kw=None, max_workers=8, lockstep=True):
    """Sequence mode on ONE GPU (BASELINE.json config C5: several independent sequences per GPU).  `sequences` is a list of
    lists of uint8 frames; returns per sequence the list of StepOut tuples (prev_xy, cur_xy, ids), identical to running
    them one by one.

    lockstep (default, sequences of equal length and frame size): one sfmgpu_multitracker advances all sequences with ONE
    batched launch per stage and step.  Otherwise every sequence gets its own context (= its own CUDA stream) and tracker,
    stepped from its own host thread (ctypes releases the GIL) - measured SLOWER than one by one on a B200 (driver-lock
    contention of many small launches), kept for ragged inputs."""
    import numpy as np
    import sfmgpu
    lkcfg_kw = lkcfg_kw or {}
    same = len(sequences) > 0 and len({(len(q), q[0].shape if len(q) else None) for q in sequences}) == 1
    if lockstep and same and len(sequences[0]) > 0:
        ctx = sfmgpu.Context(device)
        h, w = sequences[0][0].shape
        mt = ctx.multitracker(len(sequences), w, h, **lkcfg_kw)
        out = [[] for _ in sequences]
        for t in range(len(sequences[0])):
            got = mt.step(np.stack([q[t] for q in sequences]))
            for s in range(len(sequences)):
                out[s].append(got[s])
        mt.close()
        ctx.close()
        return out

    from concurrent.futures import ThreadPoolExecutor

    def one(seq):
        ctx = sfmgpu.Context(device)
        trk = ctx.tracker(**lkcfg_kw)
        out = [trk.step(img) for img in seq]
        del trk
        ctx.close()
        return out

    with ThreadPoolExecutor(max_workers=max(1, min(max_workers, len(sequences)))) as ex:
        return list(ex.map(one, sequences))
