"""ctypes binding of libtdoa_b200.so -- the same C ABI a cgo shim binds
(include/tdoa_b200.h; see INTEGRATION.md).  No numerics happen in this file: every
result comes from the CUDA library, and a missing library or GPU raises."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = _HERE / "libtdoa_b200.so"

MODE_SOURCE, MODE_BINARY, MODE_EXTENDED = 0, 1, 2
KIND_REF, KIND_TGT = 0, 1

PEAK_RESEARCHED, PEAK_EDGE, PEAK_BRUTE, PEAK_EMPTY = 0x1, 0x2, 0x4, 0x8
PEAK_BOUNDED = 0x20

ERRORS = {-1: "TDOA_E_INVALID", -2: "TDOA_E_NODEVICE", -3: "TDOA_E_CUDA", -4: "TDOA_E_NOMEM",
          -5: "TDOA_E_STATE", -6: "TDOA_E_SINGULAR", -7: "TDOA_E_IO"}

# every symbol include/tdoa_b200.h declares (tests check the library exports them all)
ABI_SYMBOLS = [
    "tdoa_default_config", "tdoa_create", "tdoa_destroy", "tdoa_last_error", "tdoa_host_alloc", "tdoa_host_free",
    "tdoa_load_u8", "tdoa_load_file", "tdoa_load_u8_pinned", "tdoa_load_u8_device", "tdoa_unpack", "tdoa_preprocess", "tdoa_set_channel", "tdoa_set_tgt_bounds", "tdoa_xcorr", "tdoa_xcorr_bounded", "tdoa_xcorr_device", "tdoa_xcorr_ranking", "tdoa_xcorr_windows", "tdoa_process", "tdoa_process_windows", "tdoa_window_fixes", "tdoa_process_windows_grid", "tdoa_window_fixes_grid", "tdoa_process_windows_retimed", "tdoa_closure", "tdoa_process_windows_closure", "tdoa_window_fixes_closure", "tdoa_exclude_stations", "tdoa_process_windows_exclude", "tdoa_window_fixes_exclude", "tdoa_xcorr_info", "tdoa_analyze",
    "tdoa_cross_correlate", "tdoa_baselines", "tdoa_solve", "tdoa_solve_binary", "tdoa_solve_ls", "tdoa_grid", "tdoa_grid_masked", "tdoa_get_stats", "tdoa_stream",
    "tdoa_set_stream", "tdoa_synchronize", "tdoa_selftest",
    "tdoa_comm_unique_id", "tdoa_comm_init", "tdoa_comm_rank", "tdoa_shard_windows",
]


class TdoaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERRORS.get(code, code)}: {message}")
        self.code = code
        self.message = message   # tdoa_last_error's text alone (the host mirror prints it as the reference would)


class Config(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_double), ("mode", C.c_int32), ("n_stations", C.c_int32),
        ("chunk_samples", C.c_int32), ("max_lag", C.c_int32), ("block_size", C.c_int32),
        ("sanity_lag", C.c_int32), ("fast_demod", C.c_int32), ("use_fft", C.c_int32),
        ("device", C.c_int32), ("seq_dc_limit", C.c_int32), ("copy_chunk", C.c_int32), ("guard_samples", C.c_int32), ("decimate", C.c_int32), ("serial_kinds", C.c_int32), ("n_devices", C.c_int32), ("reserved", C.c_int32 * 1),
    ]


class PeakStruct(C.Structure):
    _fields_ = [
        ("lag", C.c_int32), ("flags", C.c_uint32), ("corr", C.c_double), ("frac", C.c_float),
        ("margin", C.c_float), ("first_lag", C.c_int32), ("n_blocks", C.c_int32),
    ]


PEAK_DTYPE = np.dtype([("lag", "<i4"), ("flags", "<u4"), ("corr", "<f8"), ("frac", "<f4"), ("margin", "<f4"),
                       ("first_lag", "<i4"), ("n_blocks", "<i4")])
assert PEAK_DTYPE.itemsize == C.sizeof(PeakStruct) == 32


class SignalInfo(C.Structure):
    _fields_ = [("power0", C.c_double), ("dc_re", C.c_double), ("dc_im", C.c_double), ("power1", C.c_double),
                ("branch", C.c_int32), ("reserved", C.c_int32), ("n", C.c_int64)]


class SignalQuality(C.Structure):
    _fields_ = [("total_samples", C.c_int64), ("i_avg", C.c_double), ("q_avg", C.c_double), ("i_std", C.c_double),
                ("q_std", C.c_double), ("i_min", C.c_int32), ("i_max", C.c_int32), ("q_min", C.c_int32),
                ("q_max", C.c_int32), ("snr_db", C.c_double), ("power_db", C.c_double), ("dc_offset", C.c_double),
                ("iq_imbalance", C.c_double), ("has_clipping", C.c_int32), ("has_overload", C.c_int32),
                ("has_dead_zones", C.c_int32), ("has_noise", C.c_int32)]

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_}


class WindowOpts(C.Structure):
    _fields_ = [("dims", C.c_int32), ("min_margin", C.c_float), ("ref_max_residual", C.c_double),
                ("has_ref_tx", C.c_int32), ("has_init", C.c_int32), ("ref_tx_llh", C.c_double * 3),
                ("init_llh", C.c_double * 3)]


class ClosureOpts(C.Structure):
    _fields_ = [("max_residual", C.c_double), ("max_drop", C.c_int32), ("reserved", C.c_int32)]


def _closure_opts(closure) -> ClosureOpts:
    """closure = dict(max_residual=metres, max_drop=0); None: the inert check (max_residual = inf)"""
    c = dict(closure or {"max_residual": float("inf")})
    unknown = set(c) - {"max_residual", "max_drop"}
    if unknown or "max_residual" not in c:
        raise ValueError(f"closure takes max_residual and max_drop, got {sorted(c)}")
    return ClosureOpts(max_residual=float(c["max_residual"]), max_drop=int(c.get("max_drop", 0)))


class ExclusionOpts(C.Structure):
    _fields_ = [("max_rms", C.c_double), ("max_exclude", C.c_int32), ("reserved", C.c_int32)]


def _exclusion_opts(exclusion) -> ExclusionOpts:
    """exclusion = dict(max_rms=metres, max_exclude=1)"""
    x = dict(exclusion)
    unknown = set(x) - {"max_rms", "max_exclude"}
    if unknown or "max_rms" not in x:
        raise ValueError(f"exclusion takes max_rms and max_exclude, got {sorted(x)}")
    return ExclusionOpts(max_rms=float(x["max_rms"]), max_exclude=int(x.get("max_exclude", 1)))


class Stats(C.Structure):
    _fields_ = [
        ("launches_total", C.c_int64), ("launches_last", C.c_int64), ("ms_preprocess", C.c_float),
        ("ms_fft", C.c_float), ("ms_exact", C.c_float), ("ms_total", C.c_float), ("fft_launches", C.c_int64),
        ("ms_fft_seg", C.c_float), ("fft_pair_samples", C.c_int64), ("brute_pairs", C.c_int64),
        ("ms_demod", C.c_float), ("ms_boxcar", C.c_float), ("ms_cand", C.c_float), ("ms_fix", C.c_float),
        ("demod_launches", C.c_int64), ("demod_samples", C.c_int64),
        ("boxcar_launches", C.c_int64), ("boxcar_samples", C.c_int64),
        ("cand_launches", C.c_int64), ("cand_pair_samples", C.c_int64),
    ]


@dataclass
class Peak:
    lag: int
    corr: float
    frac: float
    flags: int
    margin: float
    first_lag: int
    n_blocks: int

    @property
    def researched(self) -> bool:
        return bool(self.flags & PEAK_RESEARCHED)

    @property
    def branches(self):
        return (self.flags >> 8) & 3, (self.flags >> 10) & 3


_lib = None


def library_path() -> Path:
    return _LIB


def load_library():
    """dlopen libtdoa_b200.so (never builds, never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB.exists():
        raise FileNotFoundError(f"{_LIB} is missing: run `python tdoa-geolocation_b200/build.py` "
                                "(there is no CPU fallback)")
    L = C.CDLL(str(_LIB))
    vp, i32, i64, f64p = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double)
    L.tdoa_default_config.argtypes = [i32, C.POINTER(Config)]
    L.tdoa_create.argtypes = [C.POINTER(vp), C.POINTER(Config)]
    L.tdoa_destroy.argtypes = [vp]
    L.tdoa_destroy.restype = None
    L.tdoa_last_error.argtypes = [vp]
    L.tdoa_last_error.restype = C.c_char_p
    L.tdoa_host_alloc.argtypes = [C.c_size_t]
    L.tdoa_host_alloc.restype = vp
    L.tdoa_host_free.argtypes = [vp]
    L.tdoa_host_free.restype = None
    L.tdoa_load_u8.argtypes = [vp, i32, vp, C.c_size_t]
    L.tdoa_load_u8_pinned.argtypes = [vp, i32, vp, C.c_size_t]
    L.tdoa_load_file.argtypes = [vp, i32, C.c_char_p, C.POINTER(i64)]
    L.tdoa_load_u8_device.argtypes = [vp, i32, vp, C.c_size_t]
    L.tdoa_unpack.argtypes = [vp, i32, i64, i64, vp]
    L.tdoa_preprocess.argtypes = [vp, i32, i32, i64, i64, vp, f64p, C.POINTER(i32)]
    L.tdoa_set_channel.argtypes = [vp, i32, vp, vp, i32]
    L.tdoa_xcorr.argtypes = [vp, i32, i64, i64, i32, i64, vp]
    L.tdoa_xcorr_bounded.argtypes = [vp, i32, i64, i64, i32, i64, vp, vp, vp]
    L.tdoa_set_tgt_bounds.argtypes = [vp, i32, C.c_double]
    L.tdoa_xcorr_info.argtypes = [vp, i32, vp, vp]
    L.tdoa_process.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.POINTER(i32), C.POINTER(i32)]
    L.tdoa_analyze.argtypes = [vp, i32, i32, vp, vp]
    L.tdoa_xcorr_device.argtypes = [vp, i32, i64, i64, i32, i64, vp]
    L.tdoa_xcorr_ranking.argtypes = [vp, i32, i64, i64, i32, i64, vp, vp]
    L.tdoa_xcorr_windows.argtypes = [vp, i64, i64, i32, i32, i64, vp, vp]
    L.tdoa_process_windows.argtypes = [vp, vp, C.POINTER(WindowOpts), i64, i64, i32, i32, i64] + [vp] * 9
    L.tdoa_window_fixes.argtypes = [vp, vp, C.POINTER(WindowOpts), i64, i64, i32, i32, i64] + [vp] * 9
    L.tdoa_process_windows_grid.argtypes = [vp, vp, C.POINTER(WindowOpts), i64, i64, i32, i32, i64] + [vp] * 13
    L.tdoa_window_fixes_grid.argtypes = [vp, vp, C.POINTER(WindowOpts), i64, i64, i32, i32, i64] + [vp] * 13
    L.tdoa_process_windows_retimed.argtypes = [vp, vp, C.POINTER(WindowOpts), i64, i64, i32, i64, i64, i64, i32, i64] + [vp] * 10
    L.tdoa_closure.argtypes = [vp, i32, vp, vp, i32, i32, i32, C.POINTER(ClosureOpts), vp, vp, vp]
    L.tdoa_process_windows_closure.argtypes = ([vp, vp, C.POINTER(WindowOpts), C.POINTER(ClosureOpts), i64, i64, i32, i64, i64,
                                                i64, i32, i64, i32] + [vp] * 16)
    L.tdoa_window_fixes_closure.argtypes = [vp, vp, C.POINTER(WindowOpts), C.POINTER(ClosureOpts), i64, i64, i32, i32, i64] + [vp] * 15
    L.tdoa_exclude_stations.argtypes = [vp, vp, i32, vp, vp, i32, i32, vp, i32, C.POINTER(ExclusionOpts)] + [vp] * 8
    L.tdoa_process_windows_exclude.argtypes = ([vp, vp, C.POINTER(WindowOpts), C.POINTER(ClosureOpts), C.POINTER(ExclusionOpts),
                                                i64, i64, i32, i64, i64, i64, i32, i64, i32] + [vp] * 19)
    L.tdoa_window_fixes_exclude.argtypes = ([vp, vp, C.POINTER(WindowOpts), C.POINTER(ClosureOpts), C.POINTER(ExclusionOpts),
                                             i64, i64, i32, i32, i64] + [vp] * 18)
    L.tdoa_cross_correlate.argtypes = [vp, vp, i64, vp, i64, C.POINTER(PeakStruct)]
    L.tdoa_baselines.argtypes = [vp, vp, i32, vp]
    L.tdoa_solve.argtypes = [vp, vp, i32, vp, i32, i32, vp, vp, vp]
    L.tdoa_solve_binary.argtypes = [vp, vp, i32, vp, i32, vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), vp]
    L.tdoa_solve_ls.argtypes = [vp, vp, i32, vp, i32, i32, vp, i32, vp, vp, vp, vp]
    L.tdoa_grid.argtypes = [vp, vp, i32, vp, vp, i32, i32, vp, vp, vp]
    L.tdoa_grid_masked.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, vp, vp, vp]
    L.tdoa_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.tdoa_stream.argtypes = [vp]
    L.tdoa_stream.restype = vp
    L.tdoa_set_stream.argtypes = [vp, vp]
    L.tdoa_synchronize.argtypes = [vp]
    L.tdoa_selftest.argtypes = [vp, i32, C.POINTER(C.c_int64)]
    L.tdoa_comm_unique_id.argtypes = [vp]
    L.tdoa_comm_init.argtypes = [vp, vp, i32, i32]
    L.tdoa_comm_rank.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.tdoa_shard_windows.argtypes = [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    _lib = L
    return L


def channel_taps(offset_hz: float, half_width_hz: float, n_taps: int = 63, fs: float = 2e6) -> np.ndarray:
    """Taps for Engine.set_channel: a Blackman-windowed sinc low-pass with unit DC gain whose -6 dB point is
    half_width_hz (the window's transition is symmetric about the sinc's cut-off), modulated to offset_hz about
    the centre tap, so the pass band is offset_hz +- half_width_hz with zero phase at its centre.  Designed in f64
    and rounded to complex64.  The transition is about +-2.75 fs / n_taps wide; the stop band lies below -60 dB."""
    if n_taps < 1 or n_taps % 2 == 0 or n_taps > 127:
        raise ValueError("n_taps must be odd, 1..127")
    c = (n_taps - 1) // 2
    k = np.arange(n_taps, dtype=np.float64) - c
    g = np.sinc(2.0 * half_width_hz / fs * k)
    if n_taps > 1:
        a = 2.0 * np.pi * np.arange(n_taps) / (n_taps - 1)
        g = g * (0.42 - 0.5 * np.cos(a) + 0.08 * np.cos(2.0 * a))
    g = g / g.sum()
    return (g * np.exp(2j * np.pi * offset_hz / fs * k)).astype(np.complex64)


def default_config(mode: int, **overrides) -> Config:
    cfg = Config()
    rc = load_library().tdoa_default_config(mode, C.byref(cfg))
    if rc:
        raise TdoaError(rc, f"bad mode {mode}")
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


def comm_unique_id() -> bytes:
    """tdoa_comm_unique_id: rank 0 makes the 128-byte id every rank passes to Engine.comm_init."""
    buf = (C.c_uint8 * 128)()
    L = load_library()
    rc = L.tdoa_comm_unique_id(C.cast(buf, C.c_void_p))
    if rc:
        raise TdoaError(rc, (L.tdoa_last_error(None) or b"").decode())
    return bytes(buf)


def shard_windows_rule(n_windows: int, rank: int, world: int, cursor: int = 0):
    """tdoa_shard_windows (host arithmetic, no GPU): (first, count) -- rank's windows are first, first + world, ..."""
    first, count = C.c_int32(), C.c_int32()
    rc = load_library().tdoa_shard_windows(n_windows, rank, world, cursor, C.byref(first), C.byref(count))
    if rc:
        raise ValueError(f"bad rank {rank} of {world} (cursor {cursor}, {n_windows} windows)")
    return first.value, count.value


class PinnedBuffer:
    """Page-locked host memory from tdoa_host_alloc, viewed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        self._lib = load_library()
        self.ptr = self._lib.tdoa_host_alloc(nbytes)
        if not self.ptr:
            raise MemoryError(f"tdoa_host_alloc({nbytes}) failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            self.array = None
            self._lib.tdoa_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def host_alloc(nbytes: int) -> PinnedBuffer:
    return PinnedBuffer(nbytes)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Engine:
    """One engine = one GPU.  Thin object wrapper over the C ABI."""

    def __init__(self, mode: int = MODE_BINARY, **overrides):
        self._lib = load_library()
        self.cfg = default_config(mode, **overrides)
        h = C.c_void_p()
        rc = self._lib.tdoa_create(C.byref(h), C.byref(self.cfg))
        if rc:
            raise TdoaError(rc, (self._lib.tdoa_last_error(None) or b"").decode())
        self._h = h
        self._keep = {}

    # -- plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._lib.tdoa_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc:
            raise TdoaError(rc, (self._lib.tdoa_last_error(self._h) or b"").decode())

    @property
    def n_stations(self) -> int:
        return self.cfg.n_stations

    @property
    def n_pairs(self) -> int:
        s = self.cfg.n_stations
        return s * (s - 1) // 2

    @property
    def stream(self) -> int:
        return self._lib.tdoa_stream(self._h) or 0

    def set_stream(self, stream_ptr: int):
        self._check(self._lib.tdoa_set_stream(self._h, C.c_void_p(stream_ptr)))

    def synchronize(self):
        self._check(self._lib.tdoa_synchronize(self._h))

    # -- more than one GPU, one process per GPU (tdoa_comm_init): xcorr over >= 2 windows becomes collective
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._check(self._lib.tdoa_comm_init(self._h, C.cast(buf, C.c_void_p), rank, world))

    def comm_rank(self):
        r, w = C.c_int32(), C.c_int32()
        self._check(self._lib.tdoa_comm_rank(self._h, C.byref(r), C.byref(w)))
        return r.value, w.value

    def selftest(self, which: int = 0) -> int:
        bad = C.c_int64(-1)
        self._check(self._lib.tdoa_selftest(self._h, which, C.byref(bad)))
        return bad.value

    def last_error(self) -> str:
        return (self._lib.tdoa_last_error(self._h) or b"").decode()

    def stats(self) -> dict:
        st = Stats()
        self._check(self._lib.tdoa_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in Stats._fields_}

    # -- loadIQData + extract* (processor.go:166-267)
    def load_u8(self, station: int, iq) -> None:
        if isinstance(iq, PinnedBuffer):
            ptr, n = C.c_void_p(iq.ptr), iq.nbytes
        else:
            iq = np.ascontiguousarray(iq, dtype=np.uint8)
            ptr, n = _ptr(iq), iq.size
        self._check(self._lib.tdoa_load_u8(self._h, station, ptr, n))

    def load_file(self, station: int, path) -> int:
        """loadIQData (processor.go:166-205): streams a .dat capture to the device; returns the sample count."""
        n = C.c_int64(0)
        self._check(self._lib.tdoa_load_file(self._h, station, str(path).encode(), C.byref(n)))
        return int(n.value)

    def load_u8_pinned(self, station: int, buf: "PinnedBuffer") -> None:
        """Lazy load from tdoa_host_alloc memory: returns at once; the copies are queued by the next
        call that needs the capture and the discriminator follows them chunk by chunk.  `buf` must
        stay unchanged until synchronize() or until both signal kinds were correlated."""
        self._keep[("pinned", station)] = buf
        self._check(self._lib.tdoa_load_u8_pinned(self._h, station, C.c_void_p(buf.ptr), buf.nbytes))

    def load_u8_ptr(self, station: int, ptr: int, nbytes: int) -> None:
        self._check(self._lib.tdoa_load_u8(self._h, station, C.c_void_p(ptr), nbytes))

    def load_u8_device(self, station: int, dev_ptr: int, nbytes: int, keep=None) -> None:
        self._keep[station] = keep
        self._check(self._lib.tdoa_load_u8_device(self._h, station, C.c_void_p(dev_ptr), nbytes))

    def unpack(self, station: int, first: int, count: int) -> np.ndarray:
        out = np.empty(count, np.complex64)
        self._check(self._lib.tdoa_unpack(self._h, station, first, count, _ptr(out)))
        return out

    # -- preprocessSignal (processor.go:469-499 / ELF 0x49cd40)
    def preprocess(self, station: int, kind: int, start: int, length: int):
        out = np.empty(length, np.complex64)
        power = C.c_double()
        branch = C.c_int32()
        self._check(self._lib.tdoa_preprocess(self._h, station, kind, start, length, _ptr(out),
                                              C.byref(power), C.byref(branch)))
        if self.cfg.mode == MODE_EXTENDED and self.cfg.decimate > 1:
            out = out[:length // self.cfg.decimate]
        return out, power.value, branch.value

    def set_channel(self, kind: int, taps) -> None:
        """Channel filter of `kind` (EXTENDED mode, tdoa_set_channel): a complex FIR over every signal's unpacked
        samples ahead of preprocessing.  taps: a real or complex 1-D array of odd length <= 127 (rounded to f32,
        e.g. channel_taps(...)), or None to clear."""
        if taps is None:
            self._check(self._lib.tdoa_set_channel(self._h, kind, None, None, 0))
            return
        t = np.asarray(taps)
        if t.ndim != 1:
            raise ValueError("taps must be a 1-D array")
        re = np.ascontiguousarray(t.real, np.float32)
        im = np.ascontiguousarray(t.imag, np.float32) if np.iscomplexobj(t) else None
        self._check(self._lib.tdoa_set_channel(self._h, kind, _ptr(re), _ptr(im) if im is not None else None, t.size))

    # -- ProcessTDOA pair loops (processor.go:816-850)
    def xcorr(self, kind: int, win_start: int = 0, win_len: int = 0, n_windows: int = 1, hop: int = 0) -> np.ndarray:
        out = np.zeros((n_windows, self.n_pairs), PEAK_DTYPE)
        self._check(self._lib.tdoa_xcorr(self._h, kind, win_start, win_len, n_windows, hop, _ptr(out)))
        return out

    def xcorr_ranking(self, kind: int, win_start: int = 0, win_len: int = 0, n_windows: int = 1, hop: int = 0):
        """xcorr plus the f32 ranking plane each FFT record's candidates came from (tdoa_xcorr_ranking): (records,
        ranking), ranking[w, p, d] the approximate correlation at lag index d (lag d in BINARY, d - max_lag / D in
        EXTENDED); NaN past the record's lags and on records without a ranking.  One GPU only."""
        if self.cfg.mode == MODE_EXTENDED:
            m = 2 * (self.cfg.max_lag // max(1, self.cfg.decimate)) + 1
        else:
            m = self.cfg.max_lag
        out = np.zeros((n_windows, self.n_pairs), PEAK_DTYPE)
        ranking = np.empty((n_windows, self.n_pairs, max(m, 0)), np.float32)
        self._check(self._lib.tdoa_xcorr_ranking(self._h, kind, win_start, win_len, n_windows, hop, _ptr(out),
                                                 _ptr(ranking)))
        return out, ranking

    def xcorr_bounded(self, kind: int, lo, hi, win_start: int = 0, win_len: int = 0, n_windows: int = 1,
                      hop: int = 0) -> np.ndarray:
        """xcorr with each record's lag searched within [lo, hi] (EXTENDED mode, tdoa_xcorr_bounded): lo, hi are
        int32 capture samples, broadcast to (n_windows, n_pairs).  Every record carries PEAK_BOUNDED; a maximum on the
        interval's boundary has PEAK_EDGE, an interval without a lag of the range gives PEAK_EMPTY."""
        shape = (n_windows, self.n_pairs)

        def i32(v, name):
            a = np.asarray(v)
            if a.dtype.kind not in "iu" or (a.size and (a.min() < -2 ** 31 or a.max() > 2 ** 31 - 1)):
                raise ValueError(f"{name} must be integers within int32")
            return np.ascontiguousarray(np.broadcast_to(a.astype(np.int32), shape))

        lo, hi = i32(lo, "lo"), i32(hi, "hi")
        out = np.zeros(shape, PEAK_DTYPE)
        self._check(self._lib.tdoa_xcorr_bounded(self._h, kind, win_start, win_len, n_windows, hop, _ptr(lo), _ptr(hi),
                                                 _ptr(out)))
        return out

    def set_tgt_bounds(self, guard) -> None:
        """Bounded TGT search in every windowed process call (EXTENDED mode, tdoa_set_tgt_bounds): each TGT lag is
        searched within the interval its pair's REF line and baseline allow, widened by `guard` samples on each side;
        None turns it off (the default)."""
        if guard is None:
            self._check(self._lib.tdoa_set_tgt_bounds(self._h, 0, 0.0))
        else:
            self._check(self._lib.tdoa_set_tgt_bounds(self._h, 1, float(guard)))

    def xcorr_windows(self, win_start: int, win_len: int, n_ref_windows: int, n_tgt_windows: int, hop: int):
        """Both pair loops over windows in one call (tdoa_xcorr_windows): (ref, tgt) tables.  On a multi-GPU
        engine the windows of both kinds are dealt as one list and the ranks meet once."""
        ref = np.zeros((n_ref_windows, self.n_pairs), PEAK_DTYPE)
        tgt = np.zeros((n_tgt_windows, self.n_pairs), PEAK_DTYPE)
        self._check(self._lib.tdoa_xcorr_windows(self._h, win_start, win_len, n_ref_windows, n_tgt_windows, hop,
                                                 _ptr(ref), _ptr(tgt)))
        return ref, tgt

    def xcorr_info(self, kind: int):
        """(signals, first_corr) of window 0 of the last xcorr(kind): what the reference prints while it
        works on a pair -- initial power, branch, DC bias, power before normalisation per station signal,
        and the first-pass peak correlation per pair."""
        sig = (SignalInfo * self.n_stations)()
        first = np.zeros(self.n_pairs, np.float64)
        self._check(self._lib.tdoa_xcorr_info(self._h, kind, C.cast(sig, C.c_void_p), _ptr(first)))
        return [{k: getattr(x, k) for k, _ in SignalInfo._fields_ if k != "reserved"} for x in sig], first

    def analyze(self, station: int, fast: bool = True):
        """Signal quality of a loaded capture, (ref, tgt) dicts: fast_analyzer.go (fast=True) or
        analyzer.go (fast=False) numbers."""
        ref, tgt = SignalQuality(), SignalQuality()
        self._check(self._lib.tdoa_analyze(self._h, station, 1 if fast else 0, C.byref(ref), C.byref(tgt)))
        return ref.as_dict(), tgt.as_dict()

    def xcorr_device(self, kind: int, dev_out_ptr: int, win_start: int = 0, win_len: int = 0, n_windows: int = 1,
                     hop: int = 0) -> None:
        self._check(self._lib.tdoa_xcorr_device(self._h, kind, win_start, win_len, n_windows, hop,
                                                C.c_void_p(dev_out_ptr)))

    # -- crossCorrelate seam (processor.go:619-643)
    def cross_correlate(self, sig1, sig2) -> Peak:
        a = np.ascontiguousarray(sig1, dtype=np.complex64)
        b = np.ascontiguousarray(sig2, dtype=np.complex64)
        pk = PeakStruct()
        self._check(self._lib.tdoa_cross_correlate(self._h, _ptr(a), a.size, _ptr(b), b.size, C.byref(pk)))
        return Peak(pk.lag, pk.corr, pk.frac, pk.flags, pk.margin, pk.first_lag, pk.n_blocks)

    # -- geodesy / solver (processor.go:125-163, 932-1045)
    def baselines(self, stations_llh) -> np.ndarray:
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        s = st.shape[0]
        out = np.zeros(s * (s - 1) // 2, np.float64)
        self._check(self._lib.tdoa_baselines(self._h, _ptr(st), s, _ptr(out)))
        return out

    def solve(self, stations_llh, range_diffs):
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64)
        single = rd.ndim == 1
        rd = rd.reshape(1, -1) if single else rd
        n, stride = rd.shape
        out = np.zeros((n, 3), np.float64)
        status = np.zeros(n, np.int32)
        iters = np.zeros(n, np.int32)
        self._check(self._lib.tdoa_solve(self._h, _ptr(st), st.shape[0], _ptr(rd), n, stride, _ptr(out),
                                         _ptr(status), _ptr(iters)))
        if single:
            return out[0], int(status[0]), int(iters[0])
        return out, status, iters

    def solve_binary(self, stations_llh, range_diffs):
        """solveTDOA of the shipped binary (tdoa_solve_binary): (llh, status, n_valid, n_iter, converged,
        trace[n_iter][5] = det, res1, res2, step, code)."""
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64).reshape(-1)
        out = np.zeros(3, np.float64)
        status, nv, ni, cv = (C.c_int32(0) for _ in range(4))
        trace = np.zeros((10, 5), np.float64)
        self._check(self._lib.tdoa_solve_binary(self._h, _ptr(st), st.shape[0], _ptr(rd), rd.size, _ptr(out),
                                                C.byref(status), C.byref(nv), C.byref(ni), C.byref(cv), _ptr(trace)))
        return out, status.value, nv.value, ni.value, bool(cv.value), trace[:ni.value]

    def process(self, stations_llh) -> dict:
        """ProcessTDOA from the pair loops to the fix in one call (processor.go:816-929), queued on the
        device without intermediate host synchronisation."""
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        if st.shape[0] != self.n_stations:
            raise ValueError(f"stations_llh has {st.shape[0]} rows, the engine holds {self.n_stations} stations")
        P = self.n_pairs
        ref, tgt = np.zeros(P, PEAK_DTYPE), np.zeros(P, PEAK_DTYPE)
        td, rd, fix = np.zeros(P, np.float64), np.zeros(P, np.float64), np.zeros(3, np.float64)
        status, iters = C.c_int32(0), C.c_int32(0)
        self._check(self._lib.tdoa_process(self._h, _ptr(st), _ptr(ref), _ptr(tgt), _ptr(td), _ptr(rd), _ptr(fix),
                                           C.byref(status), C.byref(iters)))
        return {"ref": ref, "tgt": tgt, "time_differences": td, "range_differences": rd, "position": fix,
                "status": int(status.value), "iters": int(iters.value)}

    def _window_opts(self, stations_llh, dims, min_margin, ref_max_residual, ref_tx_llh, init_llh):
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        if st.shape[0] != self.n_stations:
            raise ValueError(f"stations_llh has {st.shape[0]} rows, the engine holds {self.n_stations} stations")
        o = WindowOpts(dims=dims, min_margin=min_margin, ref_max_residual=ref_max_residual,
                       has_ref_tx=ref_tx_llh is not None, has_init=init_llh is not None)
        if ref_tx_llh is not None:
            o.ref_tx_llh[:] = [float(v) for v in ref_tx_llh]
        if init_llh is not None:
            o.init_llh[:] = [float(v) for v in init_llh]
        return st, o

    def _windows(self, fn, stations_llh, win_start, win_len, n_ref_windows, n_tgt_windows, hop, tables, dims,
                 min_margin, ref_max_residual, ref_tx_llh, init_llh, grid=None) -> dict:
        st, o = self._window_opts(stations_llh, dims, min_margin, ref_max_residual, ref_tx_llh, init_llh)
        P, nt = self.n_pairs, max(n_tgt_windows, 0)
        ref_fit, rd = np.zeros((P, 3), np.float64), np.zeros((nt, P), np.float64)
        used = np.zeros((nt, P), np.uint8)
        fix, rms = np.zeros((nt, 3), np.float64), np.zeros(nt, np.float64)
        status, iters = np.zeros(nt, np.int32), np.zeros(nt, np.int32)
        if grid is None:
            self._check(fn(self._h, _ptr(st), C.byref(o), win_start, win_len, n_ref_windows, n_tgt_windows, hop,
                           *[_ptr(t) for t in tables], _ptr(ref_fit), _ptr(rd), _ptr(used), _ptr(fix), _ptr(rms),
                           _ptr(status), _ptr(iters)))
            return {"ref_fit": ref_fit, "range_differences": rd, "pair_used": used.astype(bool), "position": fix,
                    "rms": rms, "status": status, "iters": iters}
        gd = np.ascontiguousarray(grid, dtype=np.float64).reshape(-1)
        if gd.size != 7:
            raise ValueError(f"grid must be 7 numbers (lat0, lon0, dlat, dlon, nlat, nlon, elev), got {gd.size}")
        seed, seed_cost, seed_index = np.zeros((nt, 3), np.float64), np.zeros(nt, np.float64), np.zeros(nt, np.int64)
        self._check(fn(self._h, _ptr(st), C.byref(o), win_start, win_len, n_ref_windows, n_tgt_windows, hop, _ptr(gd),
                       *[_ptr(t) for t in tables], _ptr(ref_fit), _ptr(rd), _ptr(used), _ptr(fix), _ptr(rms),
                       _ptr(status), _ptr(iters), _ptr(seed), _ptr(seed_cost), _ptr(seed_index)))
        return {"ref_fit": ref_fit, "range_differences": rd, "pair_used": used.astype(bool), "position": fix,
                "rms": rms, "status": status, "iters": iters, "seed": seed, "seed_cost": seed_cost,
                "seed_index": seed_index}

    def _closure_windows(self, fn, stations_llh, geometry, tables, retimed, dims, min_margin, ref_max_residual,
                         ref_tx_llh, init_llh, grid, closure, exclusion=None) -> dict:
        """tdoa_process_windows_closure (tables None: the call fills them) or tdoa_window_fixes_closure (tables =
        (ref, tgt) host inputs); with exclusion, fn is the matching _exclude call and closure may be None"""
        st, o = self._window_opts(stations_llh, dims, min_margin, ref_max_residual, ref_tx_llh, init_llh)
        S = self.n_stations
        c = _closure_opts(closure) if closure is not None or exclusion is None else None
        P = self.n_pairs
        (r0, rl, nr, rh), (t0, tl, nt, th) = geometry
        nt_ = max(nt, 0)
        ref_fit, rd = np.zeros((P, 3), np.float64), np.zeros((nt_, P), np.float64)
        used, resid, dropped = np.zeros((nt_, P), np.uint8), np.zeros((nt_, P), np.float64), np.zeros(nt_, np.int32)
        fix, rms = np.zeros((nt_, 3), np.float64), np.zeros(nt_, np.float64)
        status, iters = np.zeros(nt_, np.int32), np.zeros(nt_, np.int32)
        gd = None
        if grid is not None:
            gd = np.ascontiguousarray(grid, dtype=np.float64).reshape(-1)
            if gd.size != 7:
                raise ValueError(f"grid must be 7 numbers (lat0, lon0, dlat, dlon, nlat, nlon, elev), got {gd.size}")
        seed, seed_cost, seed_index = np.zeros((nt_, 3), np.float64), np.zeros(nt_, np.float64), np.zeros(nt_, np.int64)
        rounds, srms, excluded = np.zeros((nt_, S), np.uint8), np.full((nt_, S), np.nan), np.zeros(nt_, np.int32)
        checks = [_ptr(resid), _ptr(dropped)]
        opts = [None if c is None else C.byref(c)]
        if exclusion is not None:
            checks += [_ptr(rounds), _ptr(srms), _ptr(excluded)]
            opts.append(C.byref(_exclusion_opts(exclusion)))
        outs = [_ptr(ref_fit), _ptr(rd), _ptr(used), *checks, _ptr(fix), _ptr(rms), _ptr(status), _ptr(iters)]
        seeds = [_ptr(seed), _ptr(seed_cost), _ptr(seed_index)]
        out = {}
        if tables is None:
            ref_t, tgt_t = np.zeros((max(nr, 0), P), PEAK_DTYPE), np.zeros((nt_, P), PEAK_DTYPE)
            rate = np.zeros(self.n_stations, np.float64)
            self._check(fn(self._h, _ptr(st), C.byref(o), *opts, r0, rl, nr, rh, t0, tl, nt, th, int(retimed),
                           None if gd is None else _ptr(gd), _ptr(ref_t), _ptr(tgt_t), *outs, _ptr(rate), *seeds))
            out.update(ref=ref_t, tgt=tgt_t)
            if retimed:
                out["clock_rate"] = rate
        else:
            self._check(fn(self._h, _ptr(st), C.byref(o), *opts, r0, rl, nr, nt, rh, None if gd is None else _ptr(gd),
                           *[_ptr(t) for t in tables], *outs, *seeds))
        out.update({"ref_fit": ref_fit, "range_differences": rd, "pair_used": used == 1, "pair_dropped": used == 2,
                    "position": fix, "rms": rms, "status": status, "iters": iters})
        if c is not None:
            out.update(closure_residual=resid, dropped=dropped)
        if exclusion is not None:
            out.update(pair_excluded=used == 3, station_excluded=rounds, station_rms=srms, excluded=excluded)
        if gd is not None:
            out.update(seed=seed, seed_cost=seed_cost, seed_index=seed_index)
        return out

    def process_windows(self, stations_llh, win_start: int, win_len: int, n_ref_windows: int, n_tgt_windows: int,
                        hop: int, dims: int = 2, min_margin: float = 0.0, ref_max_residual: float = 0.0,
                        ref_tx_llh=None, init_llh=None, grid=None, closure=None, exclusion=None) -> dict:
        """Windowed ProcessTDOA (tdoa_process_windows): REF and TGT tables as xcorr_windows gives them, the REF
        lag's linear track per pair (ref_fit: lag at block 2's centre, drift in samples per sample, windows
        used), range differences and the used mask per (TGT window, pair), one least-squares fix per TGT window
        (status 0 ok, 1 degenerate, 2 too few measurements).  ref_tx_llh: the REF transmitter's position, whose
        geometric range difference is added back.  grid = (lat0, lon0, dlat, dlon, nlat, nlon, elev): each window's
        fix starts from the masked grid arg-min of its used pairs (tdoa_process_windows_grid); the result gains
        seed (the start cell), seed_cost and seed_index (-1 and NaN for a window with status 2).
        closure = dict(max_residual=metres, max_drop=0): each window's usable pairs are checked against each other
        first and the pairs the rest contradict are dropped (tdoa_process_windows_closure, statement in
        include/tdoa_b200.h); the result gains pair_dropped (usable but dropped), closure_residual (NaN where not
        usable) and dropped (pairs per window), and pair_used is the mask the fix read.
        exclusion = dict(max_rms=metres, max_exclude=1): after the first fix, each window whose rms exceeds max_rms
        is solved again without each station in turn and the station whose solve fits best is excluded
        (tdoa_process_windows_exclude, statement in include/tdoa_b200.h; combines with closure, which runs first, and
        grid, which seeds again); the result gains station_excluded[n_tgt][S] (0, or the round that excluded the
        station), station_rms[n_tgt][S] (first-round rms without each candidate station, NaN for the others),
        excluded (stations per window) and pair_excluded, and pair_used is the mask the fix read."""
        if closure is not None or exclusion is not None:
            g = (int(win_start), int(win_len), int(n_ref_windows), int(hop))
            fn = self._lib.tdoa_process_windows_closure if exclusion is None else self._lib.tdoa_process_windows_exclude
            return self._closure_windows(fn, stations_llh, (g, (g[0], g[1], int(n_tgt_windows), g[3])), None, 0, dims,
                                         min_margin, ref_max_residual, ref_tx_llh, init_llh, grid, closure, exclusion)
        ref = np.zeros((max(n_ref_windows, 0), self.n_pairs), PEAK_DTYPE)
        tgt = np.zeros((max(n_tgt_windows, 0), self.n_pairs), PEAK_DTYPE)
        fn = self._lib.tdoa_process_windows if grid is None else self._lib.tdoa_process_windows_grid
        out = self._windows(fn, stations_llh, win_start, win_len, n_ref_windows, n_tgt_windows, hop, (ref, tgt), dims,
                            min_margin, ref_max_residual, ref_tx_llh, init_llh, grid)
        out["ref"], out["tgt"] = ref, tgt
        return out

    def process_windows_retimed(self, stations_llh, ref, tgt, dims: int = 2, min_margin: float = 0.0,
                                ref_max_residual: float = 0.0, ref_tx_llh=None, init_llh=None, grid=None,
                                closure=None, exclusion=None) -> dict:
        """Re-timed target correlation (tdoa_process_windows_retimed): ref = (start, len, n, hop) and tgt = (start,
        len, n, hop) are the two kinds' window geometries.  The REF windows give each pair's drift line as in
        process_windows; the station clock rates fitted from those slopes re-time every TGT plane, so a TGT window
        may span the whole block without smearing its peak.  Returns process_windows' dict plus clock_rate[S]
        (samples per sample; NaN for a station without a fitted pair).  grid, closure and exclusion as process_windows
        (through tdoa_process_windows_closure, or _exclude with exclusion; without closure the closure check is
        inert)."""
        (r0, rl, nr, rh), (t0, tl, nt, th) = (tuple(int(v) for v in g) for g in (ref, tgt))
        if exclusion is not None:
            return self._closure_windows(self._lib.tdoa_process_windows_exclude, stations_llh,
                                         ((r0, rl, nr, rh), (t0, tl, nt, th)), None, 1, dims, min_margin,
                                         ref_max_residual, ref_tx_llh, init_llh, grid, closure, exclusion)
        if grid is not None or closure is not None:
            return self._closure_windows(self._lib.tdoa_process_windows_closure, stations_llh,
                                         ((r0, rl, nr, rh), (t0, tl, nt, th)), None, 1, dims, min_margin,
                                         ref_max_residual, ref_tx_llh, init_llh, grid, closure)
        st, o = self._window_opts(stations_llh, dims, min_margin, ref_max_residual, ref_tx_llh, init_llh)
        P, nt_ = self.n_pairs, max(nt, 0)
        ref_t, tgt_t = np.zeros((max(nr, 0), P), PEAK_DTYPE), np.zeros((nt_, P), PEAK_DTYPE)
        ref_fit, rd = np.zeros((P, 3), np.float64), np.zeros((nt_, P), np.float64)
        used = np.zeros((nt_, P), np.uint8)
        fix, rms = np.zeros((nt_, 3), np.float64), np.zeros(nt_, np.float64)
        status, iters = np.zeros(nt_, np.int32), np.zeros(nt_, np.int32)
        rate = np.zeros(self.n_stations, np.float64)
        self._check(self._lib.tdoa_process_windows_retimed(
            self._h, _ptr(st), C.byref(o), r0, rl, nr, rh, t0, tl, nt, th, _ptr(ref_t), _ptr(tgt_t), _ptr(ref_fit),
            _ptr(rd), _ptr(used), _ptr(fix), _ptr(rms), _ptr(status), _ptr(iters), _ptr(rate)))
        return {"ref_fit": ref_fit, "range_differences": rd, "pair_used": used.astype(bool), "position": fix,
                "rms": rms, "status": status, "iters": iters, "ref": ref_t, "tgt": tgt_t, "clock_rate": rate}

    def window_fixes(self, stations_llh, win_start: int, win_len: int, ref, tgt, hop: int, dims: int = 2,
                     min_margin: float = 0.0, ref_max_residual: float = 0.0, ref_tx_llh=None, init_llh=None,
                     grid=None, closure=None, exclusion=None) -> dict:
        """The fix stage of process_windows on given tables (tdoa_window_fixes): ref[n_ref][P], tgt[n_tgt][P] of
        PEAK_DTYPE, e.g. kept from xcorr_windows; window times come from the captures the engine holds.  grid: as
        process_windows (tdoa_window_fixes_grid); closure and exclusion: as process_windows
        (tdoa_window_fixes_closure, tdoa_window_fixes_exclude)."""
        ref = np.ascontiguousarray(ref, PEAK_DTYPE).reshape(-1, self.n_pairs)
        tgt = np.ascontiguousarray(tgt, PEAK_DTYPE).reshape(-1, self.n_pairs)
        if closure is not None or exclusion is not None:
            g = (int(win_start), int(win_len), ref.shape[0], int(hop))
            fn = self._lib.tdoa_window_fixes_closure if exclusion is None else self._lib.tdoa_window_fixes_exclude
            return self._closure_windows(fn, stations_llh, (g, (g[0], g[1], tgt.shape[0], g[3])), (ref, tgt), 0, dims,
                                         min_margin, ref_max_residual, ref_tx_llh, init_llh, grid, closure, exclusion)
        fn = self._lib.tdoa_window_fixes if grid is None else self._lib.tdoa_window_fixes_grid
        return self._windows(fn, stations_llh, win_start, win_len, ref.shape[0], tgt.shape[0], hop, (ref, tgt), dims,
                             min_margin, ref_max_residual, ref_tx_llh, init_llh, grid)

    def closure(self, n_stations: int, range_diffs, used, dims: int = 2, *, max_residual: float, max_drop: int = 0):
        """The closure check alone (tdoa_closure) over sets range_diffs[n_sets][>= P], used[n_sets][>= P] (an unused
        slot is never read).  Returns (used in {0, 1, 2} with 2 = dropped, residuals (NaN where not usable), dropped
        pairs per set); one set when range_diffs is 1-D."""
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64)
        single = rd.ndim == 1
        rd = rd.reshape(1, -1) if single else rd
        n, stride = rd.shape
        u = np.ascontiguousarray(np.asarray(used).astype(np.uint8).reshape(n, stride))
        c = _closure_opts({"max_residual": max_residual, "max_drop": max_drop})
        out, resid, dropped = np.zeros((n, stride), np.uint8), np.full((n, stride), np.nan), np.zeros(n, np.int32)
        self._check(self._lib.tdoa_closure(self._h, n_stations, _ptr(rd), _ptr(u), n, stride, dims, C.byref(c), _ptr(out),
                                           _ptr(resid), _ptr(dropped)))
        if single:
            return out[0], resid[0], int(dropped[0])
        return out, resid, dropped

    def exclude_stations(self, stations_llh, range_diffs, used, init_llh=None, dims: int = 2, *, max_rms: float,
                         max_exclude: int = 1) -> dict:
        """The station check alone (tdoa_exclude_stations) over sets range_diffs[n_sets][>= P], used[n_sets][>= P]
        (an unused slot is never read), from init_llh (one point, or one per set; None: the station mean).  Returns
        used (0, 1, or 3 = excluded with its station), station_excluded[n_sets][S] (0 or the round), station_rms,
        excluded (stations per set), position, rms, status and iters of the final fix; one set when range_diffs is
        1-D."""
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        S = st.shape[0]
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64)
        single = rd.ndim == 1
        rd = rd.reshape(1, -1) if single else rd
        n, stride = rd.shape
        u = np.ascontiguousarray(np.asarray(used).astype(np.uint8).reshape(n, stride))
        init = None
        if init_llh is not None:
            init = np.ascontiguousarray(np.broadcast_to(np.asarray(init_llh, np.float64).reshape(-1, 3), (n, 3)))
        x = _exclusion_opts({"max_rms": max_rms, "max_exclude": max_exclude})
        out = {"used": np.zeros((n, stride), np.uint8), "station_excluded": np.zeros((n, S), np.uint8),
               "station_rms": np.full((n, S), np.nan), "excluded": np.zeros(n, np.int32),
               "position": np.zeros((n, 3), np.float64), "rms": np.zeros(n, np.float64),
               "status": np.zeros(n, np.int32), "iters": np.zeros(n, np.int32)}
        self._check(self._lib.tdoa_exclude_stations(
            self._h, _ptr(st), S, _ptr(rd), _ptr(u), n, stride, None if init is None else _ptr(init), dims, C.byref(x),
            *[_ptr(out[k]) for k in ("used", "station_excluded", "station_rms", "excluded", "position", "rms", "status",
                                     "iters")]))
        return {k: v[0] for k, v in out.items()} if single else out

    def solve_ls(self, stations_llh, range_diffs, init_llh=None, dims: int = 2):
        """Levenberg-Marquardt fix over all pair range differences (engine-defined, SURVEY 8f-4).
        Returns (llh, rms_m, status, iters); arrays when range_diffs is 2-D."""
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64)
        single = rd.ndim == 1
        rd = rd.reshape(1, -1) if single else rd
        n, stride = rd.shape
        init = None
        if init_llh is not None:
            init = np.ascontiguousarray(np.broadcast_to(np.asarray(init_llh, np.float64).reshape(-1, 3), (n, 3)))
        out = np.zeros((n, 3), np.float64)
        rms = np.zeros(n, np.float64)
        status = np.zeros(n, np.int32)
        iters = np.zeros(n, np.int32)
        self._check(self._lib.tdoa_solve_ls(self._h, _ptr(st), st.shape[0], _ptr(rd), n, stride,
                                            _ptr(init) if init is not None else None, dims, _ptr(out), _ptr(rms),
                                            _ptr(status), _ptr(iters)))
        if single:
            return out[0], float(rms[0]), int(status[0]), int(iters[0])
        return out, rms, status, iters

    def grid(self, stations_llh, grid_desc, range_diffs, used=None):
        """Dense grid arg-min per set (tdoa_grid); used[set][p] (same shape as range_diffs): only the pairs with
        used != 0 enter the cost (tdoa_grid_masked; a set with no used pair gives index -1, cost and cell NaN)."""
        st = np.ascontiguousarray(stations_llh, dtype=np.float64).reshape(-1, 3)
        gd = np.ascontiguousarray(grid_desc, dtype=np.float64)
        rd = np.ascontiguousarray(range_diffs, dtype=np.float64)
        single = rd.ndim == 1
        rd = rd.reshape(1, -1) if single else rd
        n, stride = rd.shape
        out = np.zeros((n, 3), np.float64)
        cost = np.zeros(n, np.float64)
        idx = np.zeros(n, np.int64)
        if used is None:
            self._check(self._lib.tdoa_grid(self._h, _ptr(st), st.shape[0], _ptr(gd), _ptr(rd), n, stride, _ptr(out),
                                            _ptr(cost), _ptr(idx)))
        else:
            u = np.ascontiguousarray(np.asarray(used).astype(np.uint8).reshape(n, stride))
            self._check(self._lib.tdoa_grid_masked(self._h, _ptr(st), st.shape[0], _ptr(gd), _ptr(rd), _ptr(u), n, stride,
                                                   _ptr(out), _ptr(cost), _ptr(idx)))
        if single:
            return out[0], float(cost[0]), int(idx[0])
        return out, cost, idx
