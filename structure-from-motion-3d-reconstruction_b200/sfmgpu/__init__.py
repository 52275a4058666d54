"""ctypes binding of libsfmgpu.so (C ABI in include/sfmgpu.h) — plumbing for tests/, bench.py and the scheduler.

The product is the CUDA library; this module only marshals numpy arrays through the C ABI.  There is no CPU
fallback: if the library is missing or no B200 is visible, construction raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("SFMGPU_LIB") or os.path.join(_PKG, "libsfmgpu.so")  # SFMGPU_LIB: A/B builds of the same ABI

_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_vp = C.c_void_p
_i = C.c_int
_d = C.c_double
_ll = C.c_longlong

# every symbol include/sfmgpu.h declares (tests/test_abi.py checks the library exports exactly these)
SYMBOLS = [
    "sfmgpu_lkcfg_default", "sfmgpu_version", "sfmgpu_create", "sfmgpu_destroy", "sfmgpu_last_error", "sfmgpu_sync",
    "sfmgpu_launch_count", "sfmgpu_timer_start", "sfmgpu_timer_stop", "sfmgpu_flush_l2", "sfmgpu_profile", "sfmgpu_stage_times", "sfmgpu_fp64_peak", "sfmgpu_host_alloc",
    "sfmgpu_host_free", "sfmgpu_frames_create", "sfmgpu_frames_destroy", "sfmgpu_frames_upload",
    "sfmgpu_frames_upload_device", "sfmgpu_frames_synth", "sfmgpu_pyramid_build", "sfmgpu_frames_level_size",
    "sfmgpu_frames_download", "sfmgpu_corner_candidates", "sfmgpu_corners", "sfmgpu_sort_perm_desc",
    "sfmgpu_klt_track", "sfmgpu_klt_set_mode", "sfmgpu_select_set_mode", "sfmgpu_pairs_create", "sfmgpu_pairs_destroy", "sfmgpu_pair_frontend", "sfmgpu_pipeline_set", "sfmgpu_pair_frontend_host", "sfmgpu_pairs_totals",
    "sfmgpu_pairs_download", "sfmgpu_pairs_download_all", "sfmgpu_pairs_device_ptrs", "sfmgpu_tracker_create", "sfmgpu_tracker_destroy", "sfmgpu_tracker_reset",
    "sfmgpu_tracker_step", "sfmgpu_tracker_step_frames", "sfmgpu_tracker_tracks", "sfmgpu_tracker_totals",
    "sfmgpu_multitracker_create", "sfmgpu_multitracker_destroy", "sfmgpu_multitracker_step", "sfmgpu_multitracker_tracks",
    "sfmgpu_multitracker_prefetch", "sfmgpu_multitracker_step_pipelined",
    "sfmgpu_multitracker_totals",
    "sfmgpu_ransac_score", "sfmgpu_ransac_upload", "sfmgpu_ransac_score_resident", "sfmgpu_ransac_download",
    "sfmgpu_ransac_hypotheses", "sfmgpu_ransac_solve_score", "sfmgpu_solver_set_mode", "sfmgpu_global_desc32", "sfmgpu_desc_search", "sfmgpu_triangulate_dlt",
    "sfmgpu_stage_times_n", "sfmgpu_pairs_set_ransac", "sfmgpu_pairs_ransac_host_outputs", "sfmgpu_pairs_ransac",
    "sfmgpu_pairs_ransac_download", "sfmgpu_pairs_ransac_download_all", "sfmgpu_pairs_ransac_device_ptrs", "sfmgpu_ransac_sample",
    "sfmgpu_pairs_set_matches", "sfmgpu_ransac_set_early_stop", "sfmgpu_pairs_ransac_early",
    "sfmgpu_sched_shard", "sfmgpu_sched_unique_id", "sfmgpu_sched_create", "sfmgpu_sched_destroy", "sfmgpu_sched_pair_shard",
    "sfmgpu_sched_gather_pairs", "sfmgpu_frames_device_ptr", "sfmgpu_multitracker_reset",
    "sfmgpu_multitracker_set_ransac", "sfmgpu_multitracker_ransac_download_all", "sfmgpu_multitracker_ransac_early",
    "sfmgpu_pair_frontend_list", "sfmgpu_descs_create", "sfmgpu_descs_destroy", "sfmgpu_descs_compute", "sfmgpu_descs_upload",
    "sfmgpu_descs_download", "sfmgpu_descs_search",
]


class RansacCfg(C.Structure):
    """sfmgpu_ransac_cfg: the arguments of find_E_ransac(K, li, lj, iters, thr, min_inliers) plus the caller's size guard."""
    _fields_ = [("iters", _i), ("thr", _d), ("min_inliers", _i), ("min_points", _i)]


class LKCfg(C.Structure):
    """sfmgpu_lkcfg == LKConfig (cpp/src/templering_sfm.cpp:307-316)."""
    _fields_ = [("max_tracks", _i), ("min_tracks", _i), ("quality", _d), ("min_distance", _i), ("pyr_levels", _i),
                ("win_radius", _i), ("iters", _i), ("fb_thresh", _d)]


def lkcfg(**kw):
    c = LKCfg(2200, 900, 0.01, 8, 3, 5, 10, 1.0)
    for k, v in kw.items():
        if not hasattr(c, k):
            raise AttributeError(k)
        setattr(c, k, v)
    return c


class SfmGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sfmgpu error {code}: {msg}")
        self.code = code


def build_library(force=False):
    """Compile libsfmgpu.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    args = ["make", "-C", _PKG, "-s", "-j8"] + (["-B"] if force else [])
    subprocess.run(args, check=True)
    return LIB_PATH


def load_library():
    if not os.path.exists(LIB_PATH):
        raise SfmGpuError(-2, f"{LIB_PATH} is missing: build it with __graft_entry__.build() — there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    S = {
        "sfmgpu_lkcfg_default": (None, [C.POINTER(LKCfg)]),
        "sfmgpu_version": (_i, []),
        "sfmgpu_create": (_i, [_i, C.POINTER(_vp)]),
        "sfmgpu_destroy": (None, [_vp]),
        "sfmgpu_last_error": (C.c_char_p, [_vp]),
        "sfmgpu_sync": (_i, [_vp]),
        "sfmgpu_launch_count": (_ll, [_vp]),
        "sfmgpu_timer_start": (_i, [_vp]),
        "sfmgpu_timer_stop": (_i, [_vp, C.POINTER(C.c_float)]),
        "sfmgpu_flush_l2": (_i, [_vp, C.c_size_t]),
        "sfmgpu_profile": (_i, [_vp, _i]),
        "sfmgpu_stage_times": (_i, [_vp, C.POINTER(C.c_float)]),
        "sfmgpu_fp64_peak": (_i, [_vp, C.POINTER(_d)]),
        "sfmgpu_host_alloc": (_i, [_vp, C.c_size_t, C.POINTER(_vp)]),
        "sfmgpu_host_free": (_i, [_vp, _vp]),
        "sfmgpu_frames_create": (_i, [_vp, _i, _i, _i, _i, C.POINTER(_vp)]),
        "sfmgpu_frames_destroy": (None, [_vp, _vp]),
        "sfmgpu_frames_upload": (_i, [_vp, _vp, _i, _i, _vp]),
        "sfmgpu_frames_upload_device": (_i, [_vp, _vp, _i, _i, _vp, C.c_size_t]),
        "sfmgpu_frames_synth": (_i, [_vp, _vp, _i, _i, C.c_uint32, _i]),
        "sfmgpu_pyramid_build": (_i, [_vp, _vp, _i, _i]),
        "sfmgpu_frames_level_size": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i)]),
        "sfmgpu_frames_download": (_i, [_vp, _vp, _i, _i, _u8p]),
        "sfmgpu_corner_candidates": (_i, [_vp, _vp, _i, _d, _i32p, _f64p, _i, C.POINTER(_i), C.POINTER(_d)]),
        "sfmgpu_corners": (_i, [_vp, _vp, _i, _i, _d, _i, _f64p, C.POINTER(_i)]),
        "sfmgpu_sort_perm_desc": (_i, [_vp, _f64p, _i, _i32p]),
        "sfmgpu_klt_track": (_i, [_vp, _vp, _i, _i, _f64p, _i, _i, _i, _f64p, _f64p, _vp]),
        "sfmgpu_klt_set_mode": (_i, [_vp, _i]),
        "sfmgpu_select_set_mode": (_i, [_vp, _i]),
        "sfmgpu_pairs_create": (_i, [_vp, _i, _i, C.POINTER(_vp)]),
        "sfmgpu_pairs_destroy": (None, [_vp, _vp]),
        "sfmgpu_pair_frontend": (_i, [_vp, _vp, _i, _i, C.POINTER(LKCfg), _vp]),
        "sfmgpu_pipeline_set": (_i, [_vp, _i]),
        "sfmgpu_pair_frontend_host": (_i, [_vp, _vp, _vp, _i, C.POINTER(LKCfg), _vp, _i, _vp, _vp, _vp, _vp]),
        "sfmgpu_pairs_totals": (_i, [_vp, _vp, C.POINTER(_ll), C.POINTER(_ll), C.POINTER(_ll)]),
        "sfmgpu_pairs_download": (_i, [_vp, _vp, _i, _f64p, _f64p, _i, C.POINTER(_i), C.POINTER(_i)]),
        "sfmgpu_pairs_download_all": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_pairs_device_ptrs": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
        "sfmgpu_tracker_create": (_i, [_vp, C.POINTER(LKCfg), C.POINTER(_vp)]),
        "sfmgpu_tracker_destroy": (None, [_vp, _vp]),
        "sfmgpu_tracker_reset": (_i, [_vp, _vp, _u8p, _i, _i]),
        "sfmgpu_tracker_step": (_i, [_vp, _vp, _u8p, _i, _i, _vp, _vp, _vp, _i, C.POINTER(_i)]),
        "sfmgpu_tracker_step_frames": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _i, C.POINTER(_i)]),
        "sfmgpu_tracker_tracks": (_i, [_vp, _vp, _f64p, _i32p, _i, C.POINTER(_i)]),
        "sfmgpu_tracker_totals": (_i, [_vp, _vp, C.POINTER(_ll), C.POINTER(_ll)]),
        "sfmgpu_multitracker_create": (_i, [_vp, C.POINTER(LKCfg), _i, _i, _i, C.POINTER(_vp)]),
        "sfmgpu_multitracker_destroy": (None, [_vp, _vp]),
        "sfmgpu_multitracker_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_multitracker_prefetch": (_i, [_vp, _vp, _vp]),
        "sfmgpu_multitracker_step_pipelined": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_multitracker_tracks": (_i, [_vp, _vp, _i, _vp, _vp, _i, C.POINTER(_i)]),
        "sfmgpu_multitracker_totals": (_i, [_vp, _vp, C.POINTER(_ll), C.POINTER(_ll)]),
        "sfmgpu_ransac_score": (_i, [_vp, _f64p, _f64p, _i, _f64p, _i, _d, _vp, C.POINTER(_i), _vp, C.POINTER(_i)]),
        "sfmgpu_ransac_upload": (_i, [_vp, _f64p, _f64p, _i, _f64p, _i]),
        "sfmgpu_ransac_score_resident": (_i, [_vp, _d, C.POINTER(_i), C.POINTER(_i)]),
        "sfmgpu_ransac_download": (_i, [_vp, _vp, _vp, _i]),
        "sfmgpu_triangulate_dlt": (_i, [_vp, _f64p, _f64p, _i, _i32p, _i32p, _f64p, _f64p, _i, _f64p]),
        "sfmgpu_global_desc32": (_i, [_vp, _vp, _i, _i, _vp]),
        "sfmgpu_desc_search": (_i, [_vp, _vp, _i, _vp, _vp, C.POINTER(_i), C.POINTER(C.c_float)]),
        "sfmgpu_ransac_hypotheses": (_i, [_vp, _f64p, _f64p, _i, _i32p, _i, _vp]),
        "sfmgpu_ransac_solve_score": (_i, [_vp, _f64p, _f64p, _i, _vp, _i, _d, C.POINTER(_i), C.POINTER(_i), _vp, _vp]),
        "sfmgpu_solver_set_mode": (_i, [_vp, _i]),
        "sfmgpu_ransac_set_early_stop": (_i, [_vp, _i]),
        "sfmgpu_pairs_ransac_early": (_i, [_vp, _vp, C.POINTER(_ll)]),
        "sfmgpu_stage_times_n": (_i, [_vp, C.POINTER(C.c_float), _i]),
        "sfmgpu_pairs_set_ransac": (_i, [_vp, _vp, _vp, C.POINTER(RansacCfg)]),
        "sfmgpu_pairs_ransac_host_outputs": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_pairs_ransac": (_i, [_vp, _vp, _f64p, C.POINTER(RansacCfg), _vp]),
        "sfmgpu_pairs_ransac_download": (_i, [_vp, _vp, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), _vp, _i, _vp, _vp, _vp]),
        "sfmgpu_pairs_ransac_download_all": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_pairs_ransac_device_ptrs": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
        "sfmgpu_ransac_sample": (_i, [_vp, _i, _i, _i32p]),
        "sfmgpu_pairs_set_matches": (_i, [_vp, _vp, _i, _f64p, _f64p, _i32p]),
        "sfmgpu_frames_device_ptr": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
        "sfmgpu_multitracker_reset": (_i, [_vp, _vp]),
        "sfmgpu_multitracker_set_ransac": (_i, [_vp, _vp, _vp, C.POINTER(RansacCfg)]),
        "sfmgpu_multitracker_ransac_download_all": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "sfmgpu_multitracker_ransac_early": (_i, [_vp, _vp, C.POINTER(_ll)]),
        "sfmgpu_pair_frontend_list": (_i, [_vp, _vp, _vp, _vp, _i, C.POINTER(LKCfg), _vp]),
        "sfmgpu_descs_create": (_i, [_vp, _i, C.POINTER(_vp)]),
        "sfmgpu_descs_destroy": (None, [_vp, _vp]),
        "sfmgpu_descs_compute": (_i, [_vp, _vp, _i, _vp, _i, _i]),
        "sfmgpu_descs_upload": (_i, [_vp, _vp, _i, _i, _vp]),
        "sfmgpu_descs_download": (_i, [_vp, _vp, _i, _i, _vp]),
        "sfmgpu_descs_search": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
        "sfmgpu_sched_shard": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
        "sfmgpu_sched_unique_id": (_i, [_vp]),
        "sfmgpu_sched_create": (_i, [_vp, _i, _i, _vp, _vp, C.POINTER(_vp)]),
        "sfmgpu_sched_destroy": (None, [_vp, _vp]),
        "sfmgpu_sched_pair_shard": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
        "sfmgpu_sched_gather_pairs": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    }
    for name, (res, args) in S.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


class Context:
    """One CUDA device + stream (sfmgpu_ctx)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = _vp()
        rc = self.lib.sfmgpu_create(device, C.byref(h))
        if rc != 0:
            raise SfmGpuError(rc, "sfmgpu_create failed: no usable CUDA device (this library has no CPU fallback)")
        self.h = h
        self.device = device

    def _ck(self, rc):
        if rc != 0:
            raise SfmGpuError(rc, self.lib.sfmgpu_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.sfmgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._ck(self.lib.sfmgpu_sync(self.h))

    def launches(self):
        return int(self.lib.sfmgpu_launch_count(self.h))

    def pipeline_set(self, pairs_per_chunk):
        """Sub-chunk size of the two-lane chunk pipeline (0: sequential, one stream)."""
        self._ck(self.lib.sfmgpu_pipeline_set(self.h, pairs_per_chunk))

    def klt_set_mode(self, mode):
        """0 auto, 1 warp-per-feature kernel only, 2 lane-per-feature kernel whenever win_radius == 5."""
        self._ck(self.lib.sfmgpu_klt_set_mode(self.h, mode))

    def select_set_mode(self, mode):
        """0 radix sort + exact fallback on consumed score ties (default), 1 introsort emulation for every frame."""
        self._ck(self.lib.sfmgpu_select_set_mode(self.h, mode))

    def solver_set_mode(self, mode):
        """Device 8-point solver: 1 (default) screening solver for the counts of launches beyond one wave + Jacobi emulation
        for the winner, 0 the Jacobi emulation for every hypothesis, 2 the same through the warp-per-hypothesis kernel,
        3 screening for every launch (2, 3: tests)."""
        self._ck(self.lib.sfmgpu_solver_set_mode(self.h, mode))

    def ransac_set_early_stop(self, on):
        """Batched RANSAC stage: stop solving / scoring a pair once a hypothesis explains all of its points (default on, exact)."""
        self._ck(self.lib.sfmgpu_ransac_set_early_stop(self.h, 1 if on else 0))

    def timer_start(self):
        self._ck(self.lib.sfmgpu_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float(0)
        self._ck(self.lib.sfmgpu_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def flush_l2(self, nbytes=256 << 20):
        self._ck(self.lib.sfmgpu_flush_l2(self.h, nbytes))

    def profile(self, on=True):
        self._ck(self.lib.sfmgpu_profile(self.h, int(on)))

    def stage_times(self):
        ms = (C.c_float * 5)()
        self._ck(self.lib.sfmgpu_stage_times_n(self.h, ms, 5))
        return dict(corner_score=ms[0], corner_select=ms[1], klt=ms[2], compact=ms[3], ransac=ms[4])

    def ransac_sample(self, n, count):
        """count draws of uniform_int_distribution<int>(0, n-1) on mt19937(12345), from the device sampler."""
        out = np.zeros(max(count, 1), np.int32)
        self._ck(self.lib.sfmgpu_ransac_sample(self.h, n, count, out))
        return out[:count]

    def fp64_peak(self):
        t = _d(0)
        self._ck(self.lib.sfmgpu_fp64_peak(self.h, C.byref(t)))
        return t.value

    def pinned_empty(self, shape, dtype=np.uint8):
        """numpy array backed by page-locked host memory (freed with the context)."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = _vp()
        self._ck(self.lib.sfmgpu_host_alloc(self.h, max(n, 1), C.byref(p)))
        buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def pinned_free(self, arr):
        """Release an array obtained from pinned_empty (it must not be used afterwards)."""
        self._ck(self.lib.sfmgpu_host_free(self.h, _vp(arr.ctypes.data)))

    # ---- frames / pyramid ----------------------------------------------------------------------
    def frames(self, w, h, nframes, levels=3):
        return Frames(self, w, h, nframes, levels)

    # ---- RANSAC scoring -------------------------------------------------------------------------
    def ransac_score(self, xi, xj, E, thr, want_counts=True):
        xi = np.ascontiguousarray(xi, np.float64).reshape(-1, 2)
        xj = np.ascontiguousarray(xj, np.float64).reshape(-1, 2)
        E = np.ascontiguousarray(E, np.float64).reshape(-1, 9)
        n, H = len(xi), len(E)
        counts = np.zeros(max(H, 1), np.int32) if want_counts else None
        inl = np.zeros(max(n, 1), np.int32)
        bh, bn = _i(-1), _i(0)
        z2, z9 = np.zeros((1, 2)), np.zeros((1, 9))
        self._ck(self.lib.sfmgpu_ransac_score(self.h, xi if n else z2, xj if n else z2, n, E if H else z9, H, thr,
                                              _ptr(counts), C.byref(bh), _ptr(inl), C.byref(bn)))
        return (counts[:H] if want_counts else None), bh.value, inl[:bn.value].copy()

    def ransac_upload(self, xi, xj, E):
        xi = np.ascontiguousarray(xi, np.float64).reshape(-1, 2)
        xj = np.ascontiguousarray(xj, np.float64).reshape(-1, 2)
        E = np.ascontiguousarray(E, np.float64).reshape(-1, 9)
        self._ck(self.lib.sfmgpu_ransac_upload(self.h, xi, xj, len(xi), E, len(E)))

    def ransac_score_resident(self, thr, fetch=True):
        bh, bn = _i(-1), _i(0)
        if fetch:
            self._ck(self.lib.sfmgpu_ransac_score_resident(self.h, thr, C.byref(bh), C.byref(bn)))
            return bh.value, bn.value
        self._ck(self.lib.sfmgpu_ransac_score_resident(self.h, thr, None, None))
        return None

    def ransac_hypotheses(self, xi, xj, idx8, fetch=True):
        """Device 8-point solver (opt-in, not bit-identical to the host solver): one hypothesis per index octet; the
        points and hypotheses stay resident for ransac_score_resident / ransac_download."""
        xi = np.ascontiguousarray(xi, np.float64).reshape(-1, 2)
        xj = np.ascontiguousarray(xj, np.float64).reshape(-1, 2)
        idx8 = np.ascontiguousarray(idx8, np.int32).reshape(-1, 8)
        H = len(idx8)
        E = np.zeros((max(H, 1), 9)) if fetch else None
        self._ck(self.lib.sfmgpu_ransac_hypotheses(self.h, xi, xj, len(xi), idx8 if H else np.zeros((1, 8), np.int32), H, _ptr(E)))
        return E[:H] if fetch else None

    def ransac_solve_score(self, xi, xj, idx8, thr, iters=None):
        """Solver + scoring loop of find_E_ransac for the octets idx8 (None: `iters` octets from the reference's seeded
        sampling, drawn on the device): (winner, count, winner's E, ascending inlier list); hypotheses and counts stay
        resident (ransac_download)."""
        xi = np.ascontiguousarray(xi, np.float64).reshape(-1, 2)
        xj = np.ascontiguousarray(xj, np.float64).reshape(-1, 2)
        n = len(xi)
        if idx8 is None:
            H = int(iters)
        else:
            idx8 = np.ascontiguousarray(idx8, np.int32).reshape(-1, 8)
            H = len(idx8)
            if H == 0:
                idx8 = np.zeros((1, 8), np.int32)
        bh, bn = _i(-1), _i(0)
        E = np.zeros(9)
        inl = np.full(max(n, 1), -1, np.int32)
        self._ck(self.lib.sfmgpu_ransac_solve_score(self.h, xi, xj, n, _ptr(idx8), H, thr, C.byref(bh), C.byref(bn), _ptr(E), _ptr(inl)))
        return bh.value, bn.value, E, inl[:bn.value].copy()

    def ransac_download(self, H, n):
        counts = np.zeros(max(H, 1), np.int32)
        inl = np.full(max(n, 1), -1, np.int32)
        self._ck(self.lib.sfmgpu_ransac_download(self.h, _ptr(counts), _ptr(inl), n))
        return counts[:H], inl

    def triangulate_dlt(self, K, poses, ia, ib, ui, uj):
        poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 12)
        ia, ib = np.ascontiguousarray(ia, np.int32), np.ascontiguousarray(ib, np.int32)
        ui = np.ascontiguousarray(ui, np.float64).reshape(-1, 2)
        uj = np.ascontiguousarray(uj, np.float64).reshape(-1, 2)
        n = len(ui)
        X = np.zeros((max(n, 1), 3))
        if n:
            self._ck(self.lib.sfmgpu_triangulate_dlt(self.h, np.ascontiguousarray(K, np.float64).reshape(9), poses, len(poses), ia, ib,
                                                     ui, uj, n, X))
        return X[:n]

    def desc_search(self, descs, query, n_search=None):
        descs = np.ascontiguousarray(descs, np.float32).reshape(-1, 1024)
        query = np.ascontiguousarray(query, np.float32).reshape(1024)
        n = len(descs) if n_search is None else n_search
        scores = np.zeros(max(n, 1), np.float32)
        bid, bs = _i(-1), C.c_float(0)
        self._ck(self.lib.sfmgpu_desc_search(self.h, _ptr(descs) if len(descs) else None, n, _ptr(query), _ptr(scores),
                                             C.byref(bid), C.byref(bs)))
        return bid.value, np.float32(bs.value), scores[:n]

    def descs(self, capacity):
        """Device-resident bank of `capacity` loop-closure descriptors (zero-filled)."""
        return DescBank(self, capacity)

    def sort_perm_desc(self, keys):
        keys = np.ascontiguousarray(keys, np.float64)
        perm = np.zeros(max(len(keys), 1), np.int32)
        self._ck(self.lib.sfmgpu_sort_perm_desc(self.h, keys if len(keys) else np.zeros(1), len(keys), perm))
        return perm[:len(keys)]

    def pairs(self, max_pairs, max_corners):
        return Pairs(self, max_pairs, max_corners)

    def tracker(self, cfg=None, **kw):
        return Tracker(self, cfg if cfg is not None else lkcfg(**kw))

    def multitracker(self, n_sequences, w, h, cfg=None, **kw):
        return MultiTracker(self, n_sequences, w, h, cfg if cfg is not None else lkcfg(**kw))


class Frames:
    """sfmgpu_frames: F images of one size with their pyramids, resident in HBM."""

    def __init__(self, ctx, w, h, nframes, levels):
        self.ctx, self.w, self.h, self.n, self.levels = ctx, w, h, nframes, levels
        p = _vp()
        ctx._ck(ctx.lib.sfmgpu_frames_create(ctx.h, w, h, nframes, levels, C.byref(p)))
        self.h_ = p

    def close(self):
        if getattr(self, "h_", None) and self.ctx.h:
            self.ctx.lib.sfmgpu_frames_destroy(self.ctx.h, self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, first, imgs):
        imgs = np.ascontiguousarray(imgs, np.uint8)
        if imgs.ndim == 2:
            imgs = imgs[None]
        assert imgs.shape[1:] == (self.h, self.w), (imgs.shape, self.h, self.w)
        self.ctx._ck(self.ctx.lib.sfmgpu_frames_upload(self.ctx.h, self.h_, first, len(imgs), imgs.ctypes.data_as(_vp)))
        self._keep = imgs  # keep the host buffer alive until the stream has consumed it

    def upload_ptr(self, first, count, host_ptr):
        self.ctx._ck(self.ctx.lib.sfmgpu_frames_upload(self.ctx.h, self.h_, first, count, host_ptr))

    def synth(self, first, count, seed, t0):
        self.ctx._ck(self.ctx.lib.sfmgpu_frames_synth(self.ctx.h, self.h_, first, count, seed & 0xFFFFFFFF, t0))

    def build_pyramid(self, first=0, count=None):
        self.ctx._ck(self.ctx.lib.sfmgpu_pyramid_build(self.ctx.h, self.h_, first, self.n - first if count is None else count))

    def device_ptr(self, level=0):
        """(device address, row pitch, frame stride) of a level."""
        ptr, pitch, fs = _vp(), C.c_size_t(0), C.c_size_t(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_frames_device_ptr(self.h_, level, C.byref(ptr), C.byref(pitch), C.byref(fs)))
        return ptr.value, pitch.value, fs.value

    def level_size(self, level):
        w, h = _i(0), _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_frames_level_size(self.h_, level, C.byref(w), C.byref(h)))
        return w.value, h.value

    def download(self, frame, level=0):
        w, h = self.level_size(level)
        out = np.zeros((h, w), np.uint8) if w * h else np.zeros((h, w), np.uint8)
        if w * h:
            self.ctx._ck(self.ctx.lib.sfmgpu_frames_download(self.ctx.h, self.h_, frame, level, out))
        return out

    def candidates(self, frame, quality=0.01):
        cap = self.w * self.h
        xy = np.zeros((cap, 2), np.int32)
        s = np.zeros(cap, np.float64)
        n, mx = _i(0), _d(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_corner_candidates(self.ctx.h, self.h_, frame, quality, xy, s, cap, C.byref(n),
                                                           C.byref(mx)))
        return xy[:n.value].copy(), s[:n.value].copy(), mx.value

    def corners(self, frame, max_corners, quality=0.01, min_dist=8):
        xy = np.zeros((max(1, max_corners), 2), np.float64)
        n = _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_corners(self.ctx.h, self.h_, frame, max_corners, quality, min_dist, xy, C.byref(n)))
        return xy[:n.value].copy()

    def global_desc32(self, first, count):
        """Loop-closure descriptors (1024 floats each) of frames [first, first+count)."""
        out = np.zeros((max(count, 1), 1024), np.float32)
        self.ctx._ck(self.ctx.lib.sfmgpu_global_desc32(self.ctx.h, self.h_, first, count, _ptr(out)))
        return out[:count]

    def klt_track(self, frame_a, frame_b, p0, radius=5, iters=10, count=False):
        p0 = np.ascontiguousarray(p0, np.float64).reshape(-1, 2)
        n = len(p0)
        p1, pb = np.zeros((max(n, 1), 2)), np.zeros((max(n, 1), 2))
        nit = np.zeros(max(n, 1), np.int32)
        self.ctx._ck(self.ctx.lib.sfmgpu_klt_track(self.ctx.h, self.h_, frame_a, frame_b, p0 if n else np.zeros((1, 2)), n,
                                                   radius, iters, p1, pb, _ptr(nit)))
        return (p1[:n], pb[:n], nit[:n]) if count else (p1[:n], pb[:n])


class Pairs:
    """sfmgpu_pairs: device-resident results of a batch of frame pairs."""

    def __init__(self, ctx, max_pairs, max_corners):
        self.ctx, self.max_pairs, self.cap = ctx, max_pairs, max(1, max_corners)
        p = _vp()
        ctx._ck(ctx.lib.sfmgpu_pairs_create(ctx.h, max_pairs, max_corners, C.byref(p)))
        self.h_ = p

    def close(self):
        if getattr(self, "h_", None) and self.ctx.h:
            self.ctx.lib.sfmgpu_pairs_destroy(self.ctx.h, self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, frames, first_frame, npairs, cfg):
        self.ctx._ck(self.ctx.lib.sfmgpu_pair_frontend(self.ctx.h, frames.h_, first_frame, npairs, C.byref(cfg), self.h_))

    def run_list(self, frames, frame_a, frame_b, cfg):
        """The two-view unit over explicit frame pairs: pair k = (frame_a[k], frame_b[k]) goes to slot k."""
        fa = np.ascontiguousarray(frame_a, np.int32).reshape(-1)
        fb = np.ascontiguousarray(frame_b, np.int32).reshape(-1)
        if len(fa) != len(fb):
            raise ValueError("frame_a and frame_b differ in length")
        self.ctx._ck(self.ctx.lib.sfmgpu_pair_frontend_list(self.ctx.h, frames.h_, _ptr(fa) if len(fa) else None,
                                                            _ptr(fb) if len(fb) else None, len(fa), C.byref(cfg), self.h_))

    def run_host(self, frames, host, cfg, li=None, lj=None, nkept=None, ncorn=None, chunk=0):
        """Streaming front end over host frames [n, h, w] (uint8, ideally pinned): upload, pyramids, corners, KLT and
        the download of the results are overlapped chunk by chunk; returns when li/lj/nkept/ncorn are filled."""
        assert host.dtype == np.uint8 and host.flags["C_CONTIGUOUS"] and host.shape[1:] == (frames.h, frames.w)
        self.ctx._ck(self.ctx.lib.sfmgpu_pair_frontend_host(self.ctx.h, frames.h_, host.ctypes.data_as(_vp), host.shape[0], C.byref(cfg),
                                                            self.h_, chunk, _ptr(li), _ptr(lj), _ptr(nkept), _ptr(ncorn)))

    def totals(self):
        a, b, c = _ll(0), _ll(0), _ll(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_totals(self.ctx.h, self.h_, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def download_all(self, li, lj, nkept, ncorn):
        """Bulk D2H of the last batch into caller (ideally pinned) arrays; any may be None."""
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_download_all(self.ctx.h, self.h_, _ptr(li), _ptr(lj), _ptr(nkept), _ptr(ncorn)))

    def device_ptrs(self):
        a, b, c, d = _vp(), _vp(), _vp(), _vp()
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_device_ptrs(self.h_, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def torch_views(self, npairs):
        """Zero-copy torch views (li, lj [npairs, cap, 2] float64; n_kept, n_corners [npairs] int32) of the device results,
        for NCCL gathers by the scheduler.  Synchronise the context before handing them to another stream."""
        import torch

        class _View:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}

        li, lj, nk, nc = self.device_ptrs()
        dev = f"cuda:{self.ctx.device}"
        return (torch.as_tensor(_View(li, (npairs, self.cap, 2), "<f8"), device=dev),
                torch.as_tensor(_View(lj, (npairs, self.cap, 2), "<f8"), device=dev),
                torch.as_tensor(_View(nk, (npairs,), "<i4"), device=dev),
                torch.as_tensor(_View(nc, (npairs,), "<i4"), device=dev))

    # ---- RANSAC stage of the two-view unit (find_E_ransac per pair) ----------------------------------------------------
    def set_ransac(self, K, iters=4000, thr=2e-3, min_inliers=80, min_points=120):
        """Make find_E_ransac(K, li, lj, iters, thr, min_inliers) part of run() / run_host() (K None: off again)."""
        if K is None:
            self.ctx._ck(self.ctx.lib.sfmgpu_pairs_set_ransac(self.ctx.h, self.h_, None, None))
            return
        K = np.ascontiguousarray(K, np.float64).reshape(9)
        rc = RansacCfg(iters, thr, min_inliers, min_points)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_set_ransac(self.ctx.h, self.h_, K.ctypes.data_as(_vp), C.byref(rc)))

    def set_matches(self, li_list, lj_list):
        """Correspondences from elsewhere than the tracker: one (n_k, 2) array pair per slot; they become the last batch."""
        P = len(li_list)
        li, lj = np.zeros((max(P, 1), self.cap, 2)), np.zeros((max(P, 1), self.cap, 2))
        nk = np.zeros(max(P, 1), np.int32)
        for k, (a, b) in enumerate(zip(li_list, lj_list)):
            a, b = np.asarray(a, np.float64).reshape(-1, 2), np.asarray(b, np.float64).reshape(-1, 2)
            nk[k] = len(a)
            li[k, :len(a)], lj[k, :len(b)] = a, b
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_set_matches(self.ctx.h, self.h_, P, li, lj, nk))

    def ransac_host_outputs(self, status=None, best_n=None, inliers=None, R=None, t=None):
        self._tv_host = (status, best_n, inliers, R, t)  # keep the arrays alive
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac_host_outputs(self.ctx.h, self.h_, _ptr(status), _ptr(best_n), _ptr(inliers),
                                                                   _ptr(R), _ptr(t)))

    def ransac(self, K, iters=4000, thr=2e-3, min_inliers=80, min_points=120, E_host=None):
        """Run the stage now on the last batch.  E_host [npairs, iters, 9]: the caller's hypotheses (bit-identical path)."""
        K = np.ascontiguousarray(K, np.float64).reshape(9)
        rc = RansacCfg(iters, thr, min_inliers, min_points)
        if E_host is not None:
            E_host = np.ascontiguousarray(E_host, np.float64)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac(self.ctx.h, self.h_, K, C.byref(rc), _ptr(E_host)))

    def ransac_early(self):
        """Pairs whose scoring stopped early (a hypothesis explained all points) since the last call; resets the counter."""
        v = _ll(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac_early(self.ctx.h, self.h_, C.byref(v)))
        return int(v.value)

    def ransac_download(self, pair):
        """(status, best_h, inlier indices, E [3,3], R [3,3], t [3]) of one pair."""
        st, bh, bn = _i(0), _i(-1), _i(0)
        inl = np.zeros(self.cap, np.int32)
        E, R, t = np.zeros(9), np.zeros(9), np.zeros(3)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac_download(self.ctx.h, self.h_, pair, C.byref(st), C.byref(bh), C.byref(bn), _ptr(inl),
                                                               self.cap, _ptr(E), _ptr(R), _ptr(t)))
        return st.value, bh.value, inl[:max(bn.value, 0)].copy(), E.reshape(3, 3), R.reshape(3, 3), t

    def ransac_download_all(self, status=None, best_n=None, inliers=None, R=None, t=None):
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac_download_all(self.ctx.h, self.h_, _ptr(status), _ptr(best_n), _ptr(inliers), _ptr(R),
                                                                   _ptr(t)))

    def ransac_torch_views(self, npairs):
        """Zero-copy torch views of the stage's device results: status [npairs], best [npairs, 2] (winner, count), inliers
        [npairs, cap] (int32), R [npairs, 9], t [npairs, 3] (float64)."""
        import torch

        class _View:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}

        a, b, c, d, e = _vp(), _vp(), _vp(), _vp(), _vp()
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_ransac_device_ptrs(self.h_, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)))
        dev = f"cuda:{self.ctx.device}"
        return (torch.as_tensor(_View(a.value, (npairs,), "<i4"), device=dev), torch.as_tensor(_View(b.value, (npairs, 2), "<i4"), device=dev),
                torch.as_tensor(_View(c.value, (npairs, self.cap), "<i4"), device=dev),
                torch.as_tensor(_View(d.value, (npairs, 9), "<f8"), device=dev), torch.as_tensor(_View(e.value, (npairs, 3), "<f8"), device=dev))

    def download(self, pair):
        li, lj = np.zeros((self.cap, 2)), np.zeros((self.cap, 2))
        nk, nc = _i(0), _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_pairs_download(self.ctx.h, self.h_, pair, li, lj, self.cap, C.byref(nk), C.byref(nc)))
        return li[:nk.value].copy(), lj[:nk.value].copy(), nc.value


class DescBank:
    """sfmgpu_descs: loop-closure descriptors (1024 floats each) resident on the device, searched in one launch."""

    def __init__(self, ctx, capacity):
        self.ctx, self.capacity = ctx, capacity
        p = _vp()
        ctx._ck(ctx.lib.sfmgpu_descs_create(ctx.h, capacity, C.byref(p)))
        self.h_ = p

    def close(self):
        if getattr(self, "h_", None) and self.ctx.h:
            self.ctx.lib.sfmgpu_descs_destroy(self.ctx.h, self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def compute(self, frames, first, count, slot=0):
        """global_desc_32 of frames [first, first+count) into slots [slot, slot+count) (no host round trip)."""
        self.ctx._ck(self.ctx.lib.sfmgpu_descs_compute(self.ctx.h, self.h_, slot, frames.h_, first, count))

    def upload(self, descs, slot=0):
        descs = np.ascontiguousarray(descs, np.float32).reshape(-1, 1024)
        self.ctx._ck(self.ctx.lib.sfmgpu_descs_upload(self.ctx.h, self.h_, slot, len(descs), _ptr(descs) if len(descs) else None))

    def download(self, slot=0, count=None):
        count = self.capacity - slot if count is None else count
        out = np.zeros((max(count, 1), 1024), np.float32)
        self.ctx._ck(self.ctx.lib.sfmgpu_descs_download(self.ctx.h, self.h_, slot, count, _ptr(out)))
        return out[:count]

    def search(self, query_slots, n_search, want_scores=False):
        """Candidate search of every query (:1823-1831): (best_id [nq] int32, -1 = none; best_score [nq] float32; scores
        [nq, max n_search] float32 or None)."""
        qs = np.ascontiguousarray(query_slots, np.int32).reshape(-1)
        ns = np.ascontiguousarray(n_search, np.int32).reshape(-1)
        if len(qs) != len(ns):
            raise ValueError("query_slots and n_search differ in length")
        nq = len(qs)
        ld = int(ns.max()) if nq else 0
        bid, bs = np.full(max(nq, 1), -1, np.int32), np.zeros(max(nq, 1), np.float32)
        scores = np.zeros((max(nq, 1), max(ld, 1)), np.float32) if want_scores else None
        self.ctx._ck(self.ctx.lib.sfmgpu_descs_search(self.ctx.h, self.h_, _ptr(qs) if nq else None, _ptr(ns) if nq else None, nq,
                                                      _ptr(bid), _ptr(bs), _ptr(scores)))
        return bid[:nq], bs[:nq], (scores[:nq, :ld] if want_scores else None)


class MultiTracker:
    """sfmgpu_multitracker: S KLTTracker twins advanced in lock step (one batched launch per stage and step)."""

    def __init__(self, ctx, n_sequences, w, h, cfg):
        self.ctx, self.cfg, self.S, self.w, self.h = ctx, cfg, n_sequences, w, h
        p = _vp()
        ctx._ck(ctx.lib.sfmgpu_multitracker_create(ctx.h, C.byref(cfg), n_sequences, w, h, C.byref(p)))
        self.h_ = p
        self.cap = max(1, cfg.max_tracks, cfg.min_tracks) + 1
        self.prev = ctx.pinned_empty((n_sequences, self.cap, 2), np.float64)
        self.cur = ctx.pinned_empty((n_sequences, self.cap, 2), np.float64)
        self.ids = ctx.pinned_empty((n_sequences, self.cap), np.int32)
        self.n = np.zeros(n_sequences, np.int32)

    def close(self):
        if getattr(self, "h_", None) and self.ctx.h:
            self.ctx.lib.sfmgpu_multitracker_destroy(self.ctx.h, self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _frames(self, imgs):
        if imgs is None:
            return None
        imgs = np.ascontiguousarray(imgs, np.uint8)
        assert imgs.shape == (self.S, self.h, self.w)
        return imgs

    def prefetch(self, imgs):
        """Start uploading the frames of the next step (page-locked memory for the overlap); step(None, ...) consumes them."""
        self._pf = self._frames(imgs)  # keep the buffer alive while the copy runs
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_prefetch(self.ctx.h, self.h_, _ptr(self._pf)))

    def step(self, imgs, fetch=True, next_imgs=None):
        """imgs: [S, h, w] uint8, the next frame of every sequence (None: the prefetched ones); next_imgs: the frames of
        the following step, uploaded while this one computes.  Returns per sequence (prev_xy, cur_xy, ids) of the
        survivors (copies), or the survivor counts when fetch is False."""
        imgs, self._pf = self._frames(imgs), self._frames(next_imgs)
        a = (self.prev, self.cur, self.ids) if fetch else (None, None, None)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_step_pipelined(self.ctx.h, self.h_, _ptr(imgs), _ptr(self._pf), _ptr(a[0]), _ptr(a[1]),
                                                                     _ptr(a[2]), self.n.ctypes.data_as(_vp)))
        if not fetch:
            return self.n.copy()
        return [(self.prev[s, :self.n[s]].copy(), self.cur[s, :self.n[s]].copy(), self.ids[s, :self.n[s]].copy()) for s in range(self.S)]

    def step_ptr(self, ptr, next_ptr=None, fetch=False):
        """step() on raw addresses ([S, h, w] uint8 each; host - ideally pinned - or device memory of this GPU)."""
        a = (self.prev, self.cur, self.ids) if fetch else (None, None, None)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_step_pipelined(self.ctx.h, self.h_, _vp(ptr) if ptr else None,
                                                                     _vp(next_ptr) if next_ptr else None, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]),
                                                                     self.n.ctypes.data_as(_vp)))
        if not fetch:
            return self.n
        return [(self.prev[s, :self.n[s]].copy(), self.cur[s, :self.n[s]].copy(), self.ids[s, :self.n[s]].copy()) for s in range(self.S)]

    def reset(self):
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_reset(self.ctx.h, self.h_))

    # ---- RANSAC stage: find_E_ransac(K, prev_pts, cur_pts, ...) on every sequence's survivors inside the step -------------
    def set_ransac(self, K, iters=2500, thr=1e-3, min_inliers=60, min_points=1):
        """Make find_E_ransac(K, prev_pts, cur_pts, iters, thr, min_inliers) part of every later step (K None: off again);
        min_points=1 skips sequences without survivors, as the reference's `prev_pts.empty()` guard does."""
        if K is None:
            self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_set_ransac(self.ctx.h, self.h_, None, None))
            return
        K = np.ascontiguousarray(K, np.float64).reshape(9)
        rc = RansacCfg(iters, thr, min_inliers, min_points)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_set_ransac(self.ctx.h, self.h_, K.ctypes.data_as(_vp), C.byref(rc)))

    def ransac_results(self):
        """Results of the last step: status [S] (SKIPPED 0 / NONE 1 / OK 2), best_n [S], per sequence its ascending inlier
        indices into that step's survivors, R [S, 3, 3] and t [S, 3] (valid where status is OK)."""
        S = self.S
        st, bn = np.zeros(S, np.int32), np.zeros(S, np.int32)
        inl = np.zeros((S, self.cap), np.int32)
        R, t = np.zeros((S, 9)), np.zeros((S, 3))
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_ransac_download_all(self.ctx.h, self.h_, _ptr(st), _ptr(bn), _ptr(inl), _ptr(R),
                                                                          _ptr(t)))
        return st, bn, [inl[s, :max(bn[s], 0)].copy() for s in range(S)], R.reshape(S, 3, 3), t

    def ransac_early(self):
        """Sequences whose scoring stopped early (a hypothesis explained all survivors) since the last call; resets the counter."""
        v = _ll(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_ransac_early(self.ctx.h, self.h_, C.byref(v)))
        return int(v.value)

    def tracks(self, s):
        xy, ids = np.zeros((self.cap, 2)), np.zeros(self.cap, np.int32)
        n = _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_tracks(self.ctx.h, self.h_, s, _ptr(xy), _ptr(ids), self.cap, C.byref(n)))
        return xy[:n.value].copy(), ids[:n.value].copy()

    def totals(self):
        a, b = _ll(0), _ll(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_multitracker_totals(self.ctx.h, self.h_, C.byref(a), C.byref(b)))
        return a.value, b.value


class Tracker:
    """sfmgpu_tracker: KLTTracker twin (reset / step / tracks)."""

    def __init__(self, ctx, cfg):
        self.ctx, self.cfg = ctx, cfg
        p = _vp()
        ctx._ck(ctx.lib.sfmgpu_tracker_create(ctx.h, C.byref(cfg), C.byref(p)))
        self.h_ = p
        self.cap = max(1, cfg.max_tracks, cfg.min_tracks) + 1

    def close(self):
        if getattr(self, "h_", None) and self.ctx.h:
            self.ctx.lib.sfmgpu_tracker_destroy(self.ctx.h, self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, img):
        img = np.ascontiguousarray(img, np.uint8)
        self.ctx._ck(self.ctx.lib.sfmgpu_tracker_reset(self.ctx.h, self.h_, img, img.shape[1], img.shape[0]))

    def _outs(self, fetch):
        if not fetch:
            return None, None, None
        return np.zeros((self.cap, 2)), np.zeros((self.cap, 2)), np.zeros(self.cap, np.int32)

    def step(self, img, fetch=True):
        img = np.ascontiguousarray(img, np.uint8)
        prev, cur, ids = self._outs(fetch)
        n = _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_tracker_step(self.ctx.h, self.h_, img, img.shape[1], img.shape[0], _ptr(prev),
                                                      _ptr(cur), _ptr(ids), self.cap, C.byref(n)))
        if not fetch:
            return n.value
        return prev[:n.value].copy(), cur[:n.value].copy(), ids[:n.value].copy()

    def step_frames(self, frames, frame, fetch=True):
        prev, cur, ids = self._outs(fetch)
        n = _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_tracker_step_frames(self.ctx.h, self.h_, frames.h_, frame, _ptr(prev), _ptr(cur),
                                                             _ptr(ids), self.cap, C.byref(n)))
        if not fetch:
            return n.value
        return prev[:n.value].copy(), cur[:n.value].copy(), ids[:n.value].copy()

    def tracks(self):
        xy, ids = np.zeros((self.cap, 2)), np.zeros(self.cap, np.int32)
        n = _i(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_tracker_tracks(self.ctx.h, self.h_, xy, ids, self.cap, C.byref(n)))
        return xy[:n.value].copy(), ids[:n.value].copy()

    def totals(self):
        a, b = _ll(0), _ll(0)
        self.ctx._ck(self.ctx.lib.sfmgpu_tracker_totals(self.ctx.h, self.h_, C.byref(a), C.byref(b)))
        return a.value, b.value
