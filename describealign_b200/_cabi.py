"""ctypes binding of libdescribealign_b200.so (include/describealign_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present,
every entry point raises.  The library is built in-tree by describealign_b200.build.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DAB_LIB_PATH") or os.path.join(_HERE, "libdescribealign_b200.so")   # override: kernel-variant experiments

PCM_S16, PCM_F16 = 0, 1
VIDEO, AUDIO = 0, 1

EXPORTS = [
    "dab_abi_version", "dab_device_count", "dab_create", "dab_destroy", "dab_set_option", "dab_last_error",
    "dab_pair_create", "dab_pair_destroy", "dab_pair_sync", "dab_pair_stream", "dab_pair_set_pcm",
    "dab_pair_set_features", "dab_pair_feature_lens", "dab_pair_get_features", "dab_pair_stage_a",
    "dab_pair_get_path1", "dab_pair_get_points1", "dab_pair_stage_b", "dab_pair_get_path2",
    "dab_pair_get_points2", "dab_pair_get_stats", "dab_pair_get_timings", "dab_launch_count",
    "dab_pair_stage_a_match", "dab_pair_export_points1", "dab_pair_import_points1", "dab_pair_dp1",
    "dab_alloc_pinned", "dab_free_pinned", "dab_trim_pinned", "dab_alloc_stats", "dab_host_copy",
    "dab_set_host_wait", "dab_pair_get_timeline",
    "dab_set_log10f_correction", "dab_eval_log10f",
    "dab_pair_set_gate_energy", "dab_pair_stage_b_clusters", "dab_pair_get_corridors",
    "dab_pair_stage_b_score", "dab_pair_export_quals2", "dab_pair_import_quals2", "dab_pair_dp2",
    "dab_engine_create", "dab_engine_destroy", "dab_engine_submit", "dab_engine_next", "dab_engine_submit_b",
    "dab_engine_release", "dab_engine_slot_error", "dab_engine_slot_pair", "dab_engine_counters",
    "dab_host_continuity_error", "dab_host_continuity_error_f64", "dab_host_compress_path", "dab_host_lp_assemble", "dab_host_line_clusters", "dab_host_stretch_plan",
    "dab_index_build", "dab_index_free", "dab_index_info", "dab_pair_stage_a_against",
    "dab_pcm_reader_open", "dab_pcm_reader_progress", "dab_pcm_reader_wait", "dab_pcm_reader_close", "dab_pcm_reader_copy_to_host", "dab_stretch_best_jumps",
]


class Corridor(ctypes.Structure):
    _fields_ = [("cluster", ctypes.c_int32), ("lo", ctypes.c_int32), ("hi", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("slope", ctypes.c_double), ("offset", ctypes.c_double)]


class Cluster(ctypes.Structure):
    """dab_cluster"""
    _fields_ = [("cluster", ctypes.c_int32), ("reserved", ctypes.c_int32), ("x_first", ctypes.c_double),
                ("x_last", ctypes.c_double), ("offset", ctypes.c_double), ("slope", ctypes.c_double)]


def _stage_b_args(gains, audio_stds, lines):
    """The stage-B input of a host fit as ctypes values: gain[3], audio_std[3] and the dab_cluster array
    of the line clusters [(cluster index, x_first, x_last, offset, slope), ...]."""
    g = (ctypes.c_float * 3)(*[float(x) for x in gains])
    sd = (ctypes.c_float * 3)(*[float(x) for x in audio_stds])
    arr = (Cluster * max(len(lines), 1))()
    for k, (idx, xf, xl, offset, slope) in enumerate(lines):
        arr[k] = Cluster(int(idx), 0, float(xf), float(xl), float(offset), float(slope))
    return g, sd, arr


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int64) for n in (
        "n_video_frames", "n_audio_frames", "n_video_selected", "n_audio_queries", "n_table_entries",
        "n_enumerated", "n_candidates", "n_points1", "n_path1", "n_points2", "n_path2",
        "n_dp2_queries", "n_dp2_refills", "n_dp2_neighbour", "n_dp2_run_points")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class Job(ctypes.Structure):
    """dab_job"""
    _fields_ = [("tag", ctypes.c_uint64), ("pcm", ctypes.c_void_p * 2), ("samples", ctypes.c_int64 * 2),
                ("channels", ctypes.c_int32 * 2), ("format", ctypes.c_int32), ("on_device", ctypes.c_int32)]


class Event(ctypes.Structure):
    """dab_event"""
    _fields_ = [("kind", ctypes.c_int32), ("slot", ctypes.c_int32), ("tag", ctypes.c_uint64),
                ("status", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("n_path1", ctypes.c_int64), ("path_x", ctypes.c_void_p), ("path_y", ctypes.c_void_p),
                ("features", (ctypes.c_void_p * 3) * 2), ("feature_len", (ctypes.c_int64 * 3) * 2),
                ("n_path2", ctypes.c_int64), ("rows", ctypes.c_void_p), ("stats", Stats),
                ("timings_ms", ctypes.c_float * 16)]


class StageBIn(ctypes.Structure):
    """dab_stage_b_in"""
    _fields_ = [("gain", ctypes.c_float * 3), ("audio_std", ctypes.c_float * 3),
                ("n_audio", ctypes.c_int64), ("n_video", ctypes.c_int64),
                ("n_clusters", ctypes.c_int32), ("clusters", ctypes.c_void_p)]


EVENT_STAGE_A, EVENT_STAGE_B = 1, 2
E_TIMEOUT = 6

TIMING_SLOTS = ("features_video", "features_audio", "prep_codes", "tables", "gate", "score",
                "dp1_trace", "corridors", "dp2_trace", "dp2",
                "host_in_set_pcm", "host_in_stage_a", "host_in_stage_b", "host_in_get")

_lib = None


class DabError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the CUDA library; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise DabError(
            f"{LIB_PATH} is missing: build it with `python -m describealign_b200.build` "
            "(nvcc, sm_100a). describealign_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.dab_abi_version.restype = i32
    lib.dab_alloc_pinned.argtypes = [ctypes.c_size_t]
    lib.dab_alloc_pinned.restype = vp
    lib.dab_free_pinned.argtypes = [vp]
    lib.dab_free_pinned.restype = None
    lib.dab_trim_pinned.restype = None
    lib.dab_host_copy.argtypes = [vp, vp, ctypes.c_size_t]
    lib.dab_host_copy.restype = None
    lib.dab_alloc_stats.argtypes = [ctypes.POINTER(ctypes.c_int64 * 4)]
    lib.dab_alloc_stats.restype = None
    lib.dab_device_count.restype = i32
    pd, pl, pi32 = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32)
    lib.dab_pcm_reader_open.argtypes = [vp, i32, i64, ctypes.POINTER(vp)]
    lib.dab_pcm_reader_progress.argtypes = [vp]
    lib.dab_pcm_reader_progress.restype = i64
    lib.dab_pcm_reader_wait.argtypes = [vp, ctypes.POINTER(vp), pl]
    lib.dab_stretch_best_jumps.argtypes = [vp, vp, i32, i64, i32, vp, i32, vp, vp]
    lib.dab_pcm_reader_copy_to_host.argtypes = [vp, vp, i64]
    lib.dab_pcm_reader_close.argtypes = [vp]
    lib.dab_pcm_reader_close.restype = None
    lib.dab_host_continuity_error.argtypes = [vp, vp, i64, i32, vp]
    lib.dab_host_continuity_error_f64.argtypes = [vp, vp, vp, vp, i64, i32, vp]
    lib.dab_host_compress_path.argtypes = [vp, vp, i64, vp, vp, pl]
    lib.dab_host_lp_assemble.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, pl]
    lib.dab_host_line_clusters.argtypes = [vp, vp, vp, i64, vp, vp, vp, pl]
    lib.dab_host_stretch_plan.argtypes = [i64, i64, vp, i32, vp, vp, vp, vp, pl]
    lib.dab_set_host_wait.argtypes = [i32, i32]
    lib.dab_set_host_wait.restype = i32
    lib.dab_create.argtypes = [i32, ctypes.POINTER(vp)]
    lib.dab_destroy.argtypes = [vp]
    lib.dab_destroy.restype = None
    lib.dab_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    lib.dab_last_error.argtypes = [vp]
    lib.dab_last_error.restype = ctypes.c_char_p
    lib.dab_pair_create.argtypes = [vp, ctypes.POINTER(vp)]
    lib.dab_pair_destroy.argtypes = [vp]
    lib.dab_pair_destroy.restype = None
    lib.dab_pair_sync.argtypes = [vp]
    lib.dab_pair_stream.argtypes = [vp]
    lib.dab_pair_stream.restype = vp
    lib.dab_pair_set_pcm.argtypes = [vp, i32, vp, i64, i32, i32, i32]
    lib.dab_pair_set_features.argtypes = [vp, i32, vp, i64, vp, vp, vp, vp, i64]
    lib.dab_set_log10f_correction.argtypes = [vp, vp, ctypes.c_uint64]
    lib.dab_eval_log10f.argtypes = [vp, vp, vp, i64]
    lib.dab_pair_set_gate_energy.argtypes = [vp, i32, vp, i64]
    lib.dab_pair_feature_lens.argtypes = [vp, i32, ctypes.POINTER(i64 * 5)]
    lib.dab_pair_get_features.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.dab_pair_stage_a.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.dab_index_build.argtypes = [vp, ctypes.POINTER(vp)]
    lib.dab_index_free.argtypes = [vp]
    lib.dab_index_info.argtypes = [vp, ctypes.POINTER(i64 * 4)]
    lib.dab_pair_stage_a_against.argtypes = [vp, vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.dab_pair_get_path1.argtypes = [vp, vp, vp]
    lib.dab_pair_get_points1.argtypes = [vp, vp, vp, vp]
    lib.dab_pair_stage_a_match.argtypes = [vp, i64, i64, ctypes.POINTER(i64)]
    lib.dab_pair_export_points1.argtypes = [vp, vp, vp, vp, i32]
    lib.dab_pair_import_points1.argtypes = [vp, vp, vp, vp, i64, i32]
    lib.dab_pair_dp1.argtypes = [vp, ctypes.POINTER(i64)]
    lib.dab_pair_stage_b.argtypes = [vp, vp, i64, vp, i64, vp, ctypes.c_int32, ctypes.c_int32,
                                     ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.dab_pair_stage_b_clusters.argtypes = [vp, ctypes.POINTER(ctypes.c_float * 3), ctypes.POINTER(ctypes.c_float * 3), i64, i64,
                                              vp, ctypes.c_int32, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.dab_pair_get_corridors.argtypes = [vp, vp, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    lib.dab_pair_stage_b_score.argtypes = [vp, ctypes.POINTER(ctypes.c_float * 3), ctypes.POINTER(ctypes.c_float * 3), i64, i64,
                                           vp, ctypes.c_int32, i64, i64, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.dab_pair_export_quals2.argtypes = [vp, vp, i64, i64, i32]
    lib.dab_pair_import_quals2.argtypes = [vp, vp, i64, i32]
    lib.dab_pair_dp2.argtypes = [vp, ctypes.POINTER(i64)]
    lib.dab_pair_get_path2.argtypes = [vp, vp]
    lib.dab_pair_get_points2.argtypes = [vp, vp, vp, vp, vp]
    lib.dab_pair_get_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    lib.dab_pair_get_timings.argtypes = [vp, ctypes.POINTER(ctypes.c_float * 16)]
    lib.dab_pair_get_timeline.argtypes = [vp, vp, ctypes.POINTER(ctypes.c_float * 9), ctypes.POINTER(ctypes.c_float * 9)]
    lib.dab_launch_count.argtypes = [vp]
    lib.dab_launch_count.restype = i64
    lib.dab_engine_create.argtypes = [vp, ctypes.c_int32, ctypes.POINTER(vp)]
    lib.dab_engine_destroy.argtypes = [vp]
    lib.dab_engine_destroy.restype = None
    lib.dab_engine_submit.argtypes = [vp, ctypes.POINTER(Job)]
    lib.dab_engine_next.argtypes = [vp, ctypes.POINTER(Event), ctypes.c_int32]
    lib.dab_engine_submit_b.argtypes = [vp, ctypes.c_int32, ctypes.POINTER(StageBIn)]
    lib.dab_engine_release.argtypes = [vp, ctypes.c_int32]
    lib.dab_engine_slot_error.argtypes = [vp, ctypes.c_int32]
    lib.dab_engine_slot_error.restype = ctypes.c_char_p
    lib.dab_engine_slot_pair.argtypes = [vp, ctypes.c_int32]
    lib.dab_engine_slot_pair.restype = vp
    lib.dab_engine_counters.argtypes = [vp, ctypes.POINTER(ctypes.c_int64 * 4)]
    lib.dab_engine_counters.restype = None
    if lib.dab_abi_version() != 2:
        raise DabError("libdescribealign_b200.so has an unexpected ABI version")
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def host_copy(dst: np.ndarray, src: np.ndarray):
    """dst[...] = src for two C-contiguous arrays of equal byte size, outside the interpreter lock
    (numpy's own copy holds it, which serialises the worker threads of a batch)."""
    if dst.nbytes != src.nbytes or not dst.flags.c_contiguous or not src.flags.c_contiguous:
        raise ValueError("host_copy needs C-contiguous arrays of equal size")
    if dst.nbytes:
        load().dab_host_copy(_ptr(dst), _ptr(src), dst.nbytes)
    return dst


def copied(src: np.ndarray) -> np.ndarray:
    return host_copy(np.empty(src.shape, src.dtype), src)


def alloc_stats() -> dict:
    out = (ctypes.c_int64 * 4)()
    load().dab_alloc_stats(ctypes.byref(out))
    return {"device_allocs": int(out[0]), "device_alloc_ms": out[1] / 1e3, "pinned_allocs": int(out[2]),
            "pinned_alloc_ms": out[3] / 1e3}


class _PinnedBlock:
    """Owner of one buffer of the library's pinned pool; returns it to the pool when the last
    numpy view of it is garbage collected."""

    def __init__(self, lib, nbytes):
        self.lib = lib
        self.ptr = lib.dab_alloc_pinned(max(int(nbytes), 1))
        if not self.ptr:
            raise DabError("dab_alloc_pinned failed (no CUDA device, or out of page-locked memory)")

    def __del__(self):
        try:
            if self.ptr:
                self.lib.dab_free_pinned(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array in page-locked host memory from the library's pool (recycled when freed)."""
    lib = load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
    nbytes = n * dtype.itemsize
    block = _PinnedBlock(lib, nbytes)
    buf = (ctypes.c_char * max(nbytes, 1)).from_address(block.ptr)
    buf._block = block          # the ctypes array (kept alive as the numpy base) keeps the block
    return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


def set_host_wait(device: int = -1, mode: int = 2) -> int:
    """How host threads wait for the device: 0 CUDA default (spin), 1 blocking sync, 2 query + sleep
    polling.  Call it before the first pair is created.  Returns the device's schedule flags."""
    rc = load().dab_set_host_wait(int(device), int(mode))
    if rc < 0:
        raise DabError(f"dab_set_host_wait failed ({rc}): no usable CUDA device? (describealign_b200 has no CPU fallback)")
    return rc


class Context:
    """One per process and GPU (dab_ctx)."""

    def __init__(self, device: int = -1):
        self.lib = load()
        h = ctypes.c_void_p()
        rc = self.lib.dab_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise DabError(f"dab_create failed ({rc}): {self.lib.dab_last_error(None).decode()}")
        self.handle = h

    def check(self, rc: int):
        if rc != 0:
            raise DabError(f"describealign_b200 error {rc}: {self.lib.dab_last_error(self.handle).decode()}")

    def set_option(self, name: str, value: int):
        self.check(self.lib.dab_set_option(self.handle, name.encode(), int(value)))

    def eval_log10f(self, x: np.ndarray) -> np.ndarray:
        """The feature kernel's log10f on float32 values >= 1 (glibc's formula + the uploaded correction)."""
        x = np.ascontiguousarray(x, np.float32)
        y = np.empty_like(x)
        self.check(self.lib.dab_eval_log10f(self.handle, _ptr(x), _ptr(y), x.size))
        return y

    def set_log10f_correction(self, nibbles: np.ndarray | None, count: int = 0):
        if nibbles is None or count == 0:
            self.check(self.lib.dab_set_log10f_correction(self.handle, None, 0))
        else:
            nibbles = np.ascontiguousarray(nibbles, np.uint8)
            self.check(self.lib.dab_set_log10f_correction(self.handle, _ptr(nibbles), int(count)))

    def launches(self) -> int:
        return int(self.lib.dab_launch_count(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dab_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Index:
    """The video side of stage A of one video track (dab_index), built from `pair`'s VIDEO track and then
    read-only: any number of pairs on their own streams and threads run stage_a_against it at once."""

    def __init__(self, pair: "Pair"):
        self.ctx = pair.ctx
        self.lib = pair.lib
        h = ctypes.c_void_p()
        self.ctx.check(self.lib.dab_index_build(pair.handle, ctypes.byref(h)))
        self.handle = h

    def info(self) -> dict:
        out = (ctypes.c_int64 * 4)()
        self.ctx.check(self.lib.dab_index_info(self.handle, ctypes.byref(out)))
        return dict(n_video_frames=out[0], n_video_selected=out[1], n_table_entries=out[2], users=out[3])

    def free(self):
        """Raises DabError (and frees nothing) while a stage_a_against call on the index is running."""
        if getattr(self, "handle", None):
            self.ctx.check(self.lib.dab_index_free(self.handle))
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Pair:
    """Device-resident state of one (video, description) pair (dab_pair)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.lib = ctx.lib
        h = ctypes.c_void_p()
        ctx.check(self.lib.dab_pair_create(ctx.handle, ctypes.byref(h)))
        self.handle = h
        self._keep = []
        self._pin = {}      # name -> pinned uint8 staging buffer owned by this pair (grown, never shrunk)

    def _staging(self, name: str, shape, dtype) -> np.ndarray:
        """View of this pair's page-locked staging buffer `name`.  The buffers persist for the
        life of the pair, so a batch in steady state never calls cudaHostAlloc (which waits for
        every kernel on the device); a view is valid until the next call that reuses its name."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
        nbytes = n * dtype.itemsize
        buf = self._pin.get(name)
        if buf is None or buf.nbytes < nbytes:
            buf = pinned_empty(max(nbytes + nbytes // 4, 4096), np.uint8)
            self._pin[name] = buf
        return buf[:nbytes].view(dtype).reshape(shape)

    # ---- features -------------------------------------------------------------------------
    def set_pcm(self, track: int, pcm: np.ndarray):
        """pcm: int16 (S, ch) / (S,) interleaved samples, or float16 of the same layout."""
        if pcm.ndim == 1:
            pcm = pcm[:, None]
        if pcm.dtype == np.int16:
            fmt = PCM_S16
        elif pcm.dtype == np.float16:
            fmt = PCM_F16
        else:
            raise TypeError("PCM must be int16 or float16")
        pcm = np.ascontiguousarray(pcm)
        self._keep.append(pcm)   # the copy is asynchronous for pinned memory
        self.ctx.check(self.lib.dab_pair_set_pcm(self.handle, track, _ptr(pcm), pcm.shape[0], pcm.shape[1], fmt, 0))

    def set_pcm_device(self, track: int, dev_ptr: int, samples: int, channels: int, fmt: int = PCM_S16):
        self.ctx.check(self.lib.dab_pair_set_pcm(self.handle, track, ctypes.c_void_p(dev_ptr), samples, channels, fmt, 1))

    def set_features(self, track: int, features):
        e, z, b0, b1, b2 = features
        e = np.ascontiguousarray(e, np.float32); z = np.ascontiguousarray(z, np.float32)
        b0 = np.ascontiguousarray(b0, np.float32); b1 = np.ascontiguousarray(b1, np.float32)
        b2 = np.ascontiguousarray(b2, np.float64)
        n = min(len(z), len(b0), len(b1), len(b2))
        if not (len(z) == len(b0) == len(b1) == len(b2)) or len(e) not in (n, n + 1):
            raise ValueError("feature lengths must be n (zero crossings, bands) and n or n + 1 (energy)")
        self.ctx.check(self.lib.dab_pair_set_features(self.handle, track, _ptr(e), len(e), _ptr(z), _ptr(b0),
                                                      _ptr(b1), _ptr(b2), n))

    def set_gate_energy(self, track: int, energy):
        """The separate *_energy argument of align() (decides the not-quiet frames) when it is not features[0]."""
        e = np.ascontiguousarray(energy, np.float32)
        self.ctx.check(self.lib.dab_pair_set_gate_energy(self.handle, track, _ptr(e), len(e)))

    def feature_lens(self, track: int):
        lens = (ctypes.c_int64 * 5)()
        self.ctx.check(self.lib.dab_pair_feature_lens(self.handle, track, ctypes.byref(lens)))
        return [int(x) for x in lens]

    def get_features(self, track: int, count: int = 5, copy: bool = True):
        """The first `count` feature vectors [energy, zero crossings, band 0, band 1, band 2]
        (the host fit only needs the first three, describealign.py:735).  copy=False returns views
        of this pair's pinned staging buffers, valid until the pair's next get_features call."""
        lens = (ctypes.c_int64 * 5)()
        self.ctx.check(self.lib.dab_pair_feature_lens(self.handle, track, ctypes.byref(lens)))
        dts = (np.float32, np.float32, np.float32, np.float32, np.float64)
        out = [self._staging(f"feat{track}_{k}", lens[k], dts[k]) if k < count else None for k in range(5)]
        self.ctx.check(self.lib.dab_pair_get_features(self.handle, track, *[_ptr(a) for a in out]))
        self._keep.clear()
        return [copied(a) if copy else a for a in out[:count]]

    # ---- stage A ----------------------------------------------------------------------------
    def stage_a(self):
        npts, npath = ctypes.c_int64(), ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_a(self.handle, ctypes.byref(npts), ctypes.byref(npath)))
        self._keep.clear()
        self.n_points1, self.n_path1 = npts.value, npath.value
        return npts.value, npath.value

    def stage_a_against(self, index: "Index"):
        """Stage A of this pair's description track (AUDIO) against a shared video index: only the counts
        come back (path1() copies the path on request).  Returns (n_points, n_path)."""
        npts, npath = ctypes.c_int64(), ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_a_against(self.handle, index.handle, ctypes.byref(npts), ctypes.byref(npath)))
        self._keep.clear()
        self.n_points1, self.n_path1 = npts.value, npath.value
        return npts.value, npath.value

    def path1(self):
        x = self._staging("path1_x", self.n_path1, np.int32); y = self._staging("path1_y", self.n_path1, np.int32)
        self.ctx.check(self.lib.dab_pair_get_path1(self.handle, _ptr(x), _ptr(y)))
        return x.astype(np.int64), y.astype(np.int64)

    def points1(self):
        n = self.n_points1
        i = np.empty(n, np.int32); v = np.empty(n, np.int32); q = np.empty(n, np.float64)
        self.ctx.check(self.lib.dab_pair_get_points1(self.handle, _ptr(i), _ptr(v), _ptr(q)))
        return i, v, q

    # ---- stage A in two steps (row-sharded match stage of one long pair) ------------------------
    def stage_a_match(self, row_lo: int = 0, row_hi: int = 2 ** 62):
        """prep + tables for the whole pair; gate + scoring for audio frames row_lo <= i < row_hi."""
        npts = ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_a_match(self.handle, int(row_lo), int(row_hi), ctypes.byref(npts)))
        self._keep.clear()
        self.n_points1, self.n_path1 = npts.value, 0
        return npts.value

    def export_points1_device(self, i_ptr: int, v_ptr: int, q_ptr: int):
        """Copy this pair's match points into device buffers (e.g. torch tensors used for NCCL)."""
        self.ctx.check(self.lib.dab_pair_export_points1(self.handle, ctypes.c_void_p(i_ptr), ctypes.c_void_p(v_ptr),
                                                        ctypes.c_void_p(q_ptr), 1))

    def import_points1(self, i, v, q):
        """Replace the pair's match points by host arrays sorted by (audio frame, video frame)."""
        i = np.ascontiguousarray(i, np.int32); v = np.ascontiguousarray(v, np.int32); q = np.ascontiguousarray(q, np.float64)
        if not (len(i) == len(v) == len(q)):
            raise ValueError("point arrays must have equal lengths")
        self.ctx.check(self.lib.dab_pair_import_points1(self.handle, _ptr(i), _ptr(v), _ptr(q), len(i), 0))
        self.n_points1 = len(i)

    def import_points1_device(self, i_ptr: int, v_ptr: int, q_ptr: int, n: int):
        self.ctx.check(self.lib.dab_pair_import_points1(self.handle, ctypes.c_void_p(i_ptr), ctypes.c_void_p(v_ptr),
                                                        ctypes.c_void_p(q_ptr), int(n), 1))
        self.n_points1 = int(n)

    def dp1(self):
        npath = ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_dp1(self.handle, ctypes.byref(npath)))
        self.n_path1 = npath.value
        return npath.value

    # ---- stage B ----------------------------------------------------------------------------
    def stage_b(self, audio_scaled: np.ndarray, video_scaled: np.ndarray, plans, n_clusters: int):
        if np.ndim(audio_scaled) != 2 or np.shape(audio_scaled)[1] != 3 or np.ndim(video_scaled) != 2 or \
                np.shape(video_scaled)[1] != 3:
            raise ValueError("scaled features must be (n, 3) float32")
        # staged in pinned memory: the upload is then one asynchronous DMA per array
        a = self._staging("audio_scaled", np.shape(audio_scaled), np.float32)
        v = self._staging("video_scaled", np.shape(video_scaled), np.float32)
        for dst, src in ((a, audio_scaled), (v, video_scaled)):
            if isinstance(src, np.ndarray) and src.dtype == np.float32 and src.flags.c_contiguous:
                host_copy(dst, src)
            else:
                np.copyto(dst, src, casting="same_kind")
        plans = [p for p in plans if p[2] > p[1]]
        arr = (Corridor * max(len(plans), 1))()
        for k, (idx, lo, hi, slope, offset) in enumerate(plans):
            arr[k] = Corridor(int(idx), int(lo), int(hi), 0, float(slope), float(offset))
        npts, npath = ctypes.c_int64(), ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_b(self.handle, _ptr(a), a.shape[0], _ptr(v), v.shape[0],
                                                 ctypes.cast(arr, ctypes.c_void_p), len(plans), int(n_clusters),
                                                 ctypes.byref(npts), ctypes.byref(npath)))
        self.n_points2, self.n_path2 = npts.value, npath.value
        return npts.value, npath.value

    def stage_b_clusters(self, gains, audio_stds, n_audio: int, n_video: int, lines):
        """Stage B from the host fit's line clusters [(cluster index, x_first, x_last, offset, slope), ...]:
        scaling, corridor planning (describealign.py:895-932), scoring, DP 2 and traceback on the device."""
        g, sd, arr = _stage_b_args(gains, audio_stds, lines)
        npts, npath = ctypes.c_int64(), ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_b_clusters(self.handle, ctypes.byref(g), ctypes.byref(sd), int(n_audio), int(n_video),
                                                          ctypes.cast(arr, ctypes.c_void_p), len(lines),
                                                          ctypes.byref(npts), ctypes.byref(npath)))
        self.n_points2, self.n_path2 = npts.value, npath.value
        return npts.value, npath.value

    # ---- stage B in steps (corridor rows of one long pair scored on several GPUs) -----------------
    def stage_b_score(self, gains, audio_stds, n_audio: int, n_video: int, lines, row_lo: int = 0, row_hi: int = 2 ** 62):
        """Plans the corridors and builds the whole pass-2 point list; quals only for audio rows
        [row_lo, row_hi).  Returns (n_points, first_point, n_mine): this rank's points are
        [first_point, first_point + n_mine)."""
        g, sd, arr = _stage_b_args(gains, audio_stds, lines)
        npts, first, mine = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_stage_b_score(self.handle, ctypes.byref(g), ctypes.byref(sd), int(n_audio), int(n_video),
                                                       ctypes.cast(arr, ctypes.c_void_p), len(lines), int(row_lo), int(row_hi),
                                                       ctypes.byref(npts), ctypes.byref(first), ctypes.byref(mine)))
        self.n_points2, self.n_path2 = npts.value, 0
        return npts.value, first.value, mine.value

    def export_quals2_device(self, q_ptr: int, first: int, count: int):
        self.ctx.check(self.lib.dab_pair_export_quals2(self.handle, ctypes.c_void_p(q_ptr), int(first), int(count), 1))

    def export_quals2(self, first: int, count: int) -> np.ndarray:
        q = np.empty(count, np.float64)
        self.ctx.check(self.lib.dab_pair_export_quals2(self.handle, _ptr(q), int(first), int(count), 0))
        return q

    def import_quals2_device(self, q_ptr: int, n: int):
        self.ctx.check(self.lib.dab_pair_import_quals2(self.handle, ctypes.c_void_p(q_ptr), int(n), 1))

    def import_quals2(self, q: np.ndarray):
        q = np.ascontiguousarray(q, np.float64)
        self.ctx.check(self.lib.dab_pair_import_quals2(self.handle, _ptr(q), len(q), 0))

    def dp2(self):
        npath = ctypes.c_int64()
        self.ctx.check(self.lib.dab_pair_dp2(self.handle, ctypes.byref(npath)))
        self.n_path2 = npath.value
        return npath.value

    def corridors(self):
        """The corridors of the last stage B as scored: [(cluster, lo, hi, slope, offset), ...] (empty ones
        dropped), i.e. what the reference computes in describealign.py:912-932."""
        n = ctypes.c_int32()
        self.ctx.check(self.lib.dab_pair_get_corridors(self.handle, None, 0, ctypes.byref(n)))
        arr = (Corridor * max(n.value, 1))()
        self.ctx.check(self.lib.dab_pair_get_corridors(self.handle, ctypes.cast(arr, ctypes.c_void_p), n.value, ctypes.byref(n)))
        return [(c.cluster, c.lo, c.hi, c.slope, c.offset) for c in arr[:n.value] if c.hi > c.lo]

    def path2(self):
        rows = self._staging("path2", (self.n_path2, 5), np.float64)
        self.ctx.check(self.lib.dab_pair_get_path2(self.handle, _ptr(rows)))
        return copied(rows)

    def points2(self):
        n = self.n_points2
        i = np.empty(n, np.int32); j = np.empty(n, np.float64); c = np.empty(n, np.int32); q = np.empty(n, np.float64)
        self.ctx.check(self.lib.dab_pair_get_points2(self.handle, _ptr(i), _ptr(j), _ptr(c), _ptr(q)))
        return i, j, c, q

    # ---- introspection ------------------------------------------------------------------------
    def stats(self) -> dict:
        s = Stats()
        self.ctx.check(self.lib.dab_pair_get_stats(self.handle, ctypes.byref(s)))
        return s.as_dict()

    def timings(self) -> dict:
        ms = (ctypes.c_float * 16)()
        self.ctx.check(self.lib.dab_pair_get_timings(self.handle, ctypes.byref(ms)))
        return {name: float(ms[k]) for k, name in enumerate(TIMING_SLOTS)}

    def timeline(self, ref_event: int) -> dict:
        """(start, end) of the device stages in ms after `ref_event` (a cudaEvent_t handle)."""
        t0, t1 = (ctypes.c_float * 9)(), (ctypes.c_float * 9)()
        self.ctx.check(self.lib.dab_pair_get_timeline(self.handle, ctypes.c_void_p(ref_event), ctypes.byref(t0), ctypes.byref(t1)))
        return {name: (float(t0[k]), float(t1[k])) for k, name in enumerate(TIMING_SLOTS[:9]) if t0[k] >= 0}

    def sync(self):
        self.ctx.check(self.lib.dab_pair_sync(self.handle))

    @property
    def stream(self) -> int:
        return int(self.lib.dab_pair_stream(self.handle) or 0)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dab_pair_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _view(ptr, n, dtype):
    """numpy view of n elements of page-locked memory owned by an engine slot (no copy)."""
    dtype = np.dtype(dtype)
    if not ptr or n <= 0:
        return np.empty(0, dtype)
    buf = (ctypes.c_char * (int(n) * dtype.itemsize)).from_address(int(ptr))
    return np.frombuffer(buf, dtype=dtype, count=int(n))


class Engine:
    """dab_engine: many pairs in flight on one GPU, one scheduler thread inside the library.

    submit() queues a pair; next() hands out events: EVENT_STAGE_A (pass-1 path + the features the host
    fit needs) to be answered with submit_b(), and EVENT_STAGE_B (final path rows) to be answered with
    release().  Arrays returned by the view helpers alias the slot's page-locked buffers: copy what must
    outlive the slot."""

    def __init__(self, ctx: Context, slots: int = 32):
        self.ctx = ctx
        self.lib = ctx.lib
        h = ctypes.c_void_p()
        ctx.check(self.lib.dab_engine_create(ctx.handle, int(slots), ctypes.byref(h)))
        self.handle = h
        self.slots = int(slots)
        self._keep = {}          # tag -> PCM arrays that must stay alive until stage A has consumed them

    def submit(self, tag: int, video, audio, fmt: int | None = None):
        """video / audio: interleaved (S, ch) / (S,) int16 or float16 numpy arrays (ideally page-locked),
        or (device pointer, samples per channel, channels) tuples for device-resident int16 PCM."""
        job = Job()
        job.tag = int(tag)
        on_device = isinstance(video, tuple)
        keep = []
        for t, p in enumerate((video, audio)):
            if on_device:
                ptr, samples, ch = p
                job.pcm[t] = ctypes.c_void_p(int(ptr))
                job.samples[t], job.channels[t] = int(samples), int(ch)
                f = PCM_S16 if fmt is None else fmt
            else:
                p = np.asarray(p)
                if p.ndim == 1:
                    p = p[:, None]
                if p.dtype == np.int16:
                    f = PCM_S16
                elif p.dtype == np.float16:
                    f = PCM_F16
                else:
                    raise TypeError("PCM must be int16 or float16")
                p = np.ascontiguousarray(p)
                keep.append(p)
                job.pcm[t] = p.ctypes.data_as(ctypes.c_void_p)
                job.samples[t], job.channels[t] = p.shape[0], p.shape[1]
            if t == 0:
                job.format = f
            elif f != job.format:
                raise TypeError("both tracks must have the same sample format")
        job.on_device = 1 if on_device else 0
        self._keep[int(tag)] = keep
        self.ctx.check(self.lib.dab_engine_submit(self.handle, ctypes.byref(job)))

    def next(self, timeout_ms: int = -1):
        """The next finished stage, or None after timeout_ms (0 = poll, < 0 = wait)."""
        evt = Event()
        rc = self.lib.dab_engine_next(self.handle, ctypes.byref(evt), int(timeout_ms))
        if rc == E_TIMEOUT:
            return None
        self.ctx.check(rc)
        if evt.kind == EVENT_STAGE_A:
            self._keep.pop(int(evt.tag), None)
        return evt

    def error(self, evt) -> str:
        return (self.lib.dab_engine_slot_error(self.handle, evt.slot) or b"").decode()

    # ---- views of an event's results -----------------------------------------------------------
    @staticmethod
    def path1(evt):
        return _view(evt.path_x, evt.n_path1, np.int32), _view(evt.path_y, evt.n_path1, np.int32)

    @staticmethod
    def features(evt, track: int):
        return [_view(evt.features[track][f], evt.feature_len[track][f], np.float32) for f in range(3)]

    @staticmethod
    def rows(evt):
        return _view(evt.rows, 5 * evt.n_path2, np.float64).reshape(-1, 5)

    @staticmethod
    def timings(evt) -> dict:
        return {name: float(evt.timings_ms[k]) for k, name in enumerate(TIMING_SLOTS)}

    @staticmethod
    def stage_b_struct(gains, audio_stds, n_audio: int, n_video: int, lines):
        """The dab_stage_b_in of a host fit (reusable: the engine copies the arrays on submit).
        lines: the fit's line clusters (host_fit.cluster_lines); the corridors are planned on the device."""
        b = StageBIn()
        b.gain, b.audio_std, arr = _stage_b_args(gains, audio_stds, lines)
        b.n_audio, b.n_video = int(n_audio), int(n_video)
        b.clusters = ctypes.cast(arr, ctypes.c_void_p)
        b.n_clusters = len(lines)
        b._cluster_array = arr           # keeps the array alive as long as the struct
        return b

    def submit_b(self, slot: int, gains=None, audio_stds=None, n_audio=0, n_video=0, lines=(), struct: StageBIn | None = None):
        b = struct if struct is not None else self.stage_b_struct(gains, audio_stds, n_audio, n_video, lines)
        self.ctx.check(self.lib.dab_engine_submit_b(self.handle, int(slot), ctypes.byref(b)))

    def release(self, slot: int):
        self.ctx.check(self.lib.dab_engine_release(self.handle, int(slot)))

    def counters(self) -> dict:
        out = (ctypes.c_int64 * 4)()
        self.lib.dab_engine_counters(self.handle, ctypes.byref(out))
        return {"scheduler_loops": int(out[0]), "scheduler_idle_sleeps": int(out[1])}

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dab_engine_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
