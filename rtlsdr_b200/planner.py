"""Hop planner binding: host/rtl_power_plan.c (reference src/rtl_power.c:438-540)."""
import ctypes
import os
from dataclasses import dataclass, field
from typing import List

from . import _build

RP_MAX_TUNES = 3000


class _RpPlan(ctypes.Structure):
    _fields_ = [("tune_count", ctypes.c_int), ("bin_e", ctypes.c_int), ("buf_len", ctypes.c_int),
                ("downsample", ctypes.c_int), ("downsample_passes", ctypes.c_int),
                ("rate", ctypes.c_int), ("bw_seen", ctypes.c_int), ("lower", ctypes.c_int),
                ("upper", ctypes.c_int), ("max_size", ctypes.c_int), ("crop", ctypes.c_double),
                ("bin_size", ctypes.c_double), ("freq", ctypes.c_int * RP_MAX_TUNES)]


_HOST = None


def host_library():
    """host/_build/librtlpower_host.so (planner, CSV formatter, synthetic source)."""
    global _HOST
    if _HOST is None:
        path = os.path.join(_build.HOST_BUILD, "librtlpower_host.so")
        if not os.path.exists(path):
            _build.build_host()
        L = ctypes.CDLL(path)
        L.rp_plan_range.argtypes = [ctypes.c_char_p, ctypes.c_double, ctypes.c_int, ctypes.POINTER(_RpPlan)]
        L.rp_csv_row.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(_RpPlan), ctypes.c_int,
                                 ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        L.rp_db_count.argtypes = [ctypes.POINTER(_RpPlan)]
        L.rp_csv_columns.argtypes = [ctypes.POINTER(_RpPlan), ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_void_p]
        L.rp_csv_columns.restype = None
        for fn in (L.rp_atofs, L.rp_atoft, L.rp_atofp):
            fn.argtypes = [ctypes.c_char_p]
            fn.restype = ctypes.c_double
        L.synth_generate.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t]
        L.synth_generate_cube.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                          ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int]
        L.synth_generate_cube.restype = None
        L.synth_fnv1a_int64.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint64]
        L.synth_fnv1a_int64.restype = ctypes.c_uint64
        _HOST = L
    return _HOST


@dataclass
class Plan:
    tune_count: int
    bin_e: int
    buf_len: int
    downsample: int
    downsample_passes: int
    rate: int
    crop: float
    boxcar: int
    comp_fir_size: int
    bw_seen: int = 0
    bin_size: float = 0.0
    freqs: List[int] = field(default_factory=list)
    _c: object = None

    def as_dict(self):
        return dict(tune_count=self.tune_count, bin_e=self.bin_e, buf_len=self.buf_len,
                    downsample=self.downsample, downsample_passes=self.downsample_passes,
                    rate=self.rate, crop=self.crop, boxcar=self.boxcar,
                    comp_fir_size=self.comp_fir_size, freqs=list(self.freqs))

    @property
    def db_count(self):
        return host_library().rp_db_count(ctypes.byref(self._c))

    def csv_columns(self, hops=None):
        """(low int32 [rows], high int32 [rows], step) of the rows of `hops` (default: all), the table
        GpuScan.set_csv_columns() takes (rp_csv_columns, the numbers csv_row() prints)"""
        import numpy as np
        hops = range(self.tune_count) if hops is None else hops
        low = np.zeros(len(hops), dtype=np.int32)
        high = np.zeros(len(hops), dtype=np.int32)
        lo, hi, step = ctypes.c_int(), ctypes.c_int(), ctypes.c_double()
        for i, h in enumerate(hops):
            host_library().rp_csv_columns(ctypes.byref(self._c), h, ctypes.byref(lo), ctypes.byref(hi),
                                          ctypes.byref(step))
            low[i], high[i] = lo.value, hi.value
        return low, high, step.value

    def csv_row(self, hop, samples, db):
        """'low, high, step, samples, dB...' exactly as csv_dbm prints it (rtl_power.c:739-760)."""
        import numpy as np
        db = np.ascontiguousarray(db, dtype=np.float64)
        cap = db.size * 16 + 256
        buf = ctypes.create_string_buffer(cap)
        n = host_library().rp_csv_row(buf, cap, ctypes.byref(self._c), hop, samples,
                                      db.ctypes.data, db.size)
        if n < 0:
            raise ValueError("row buffer too small")
        return buf.value.decode()


def plan_scan(freq_range, crop=0.0, fir=None):
    """frequency_range(): freq_range = 'lower:upper:bin'; fir = the -F argument or None."""
    boxcar = 1 if fir is None else 0
    c = _RpPlan()
    rc = host_library().rp_plan_range(freq_range.encode(), crop, boxcar, ctypes.byref(c))
    if rc:
        raise ValueError(f"rp_plan_range({freq_range!r}) failed: {rc}")
    return Plan(c.tune_count, c.bin_e, c.buf_len, c.downsample, c.downsample_passes, c.rate, c.crop,
                boxcar, 0 if fir is None else int(fir), c.bw_seen, c.bin_size,
                [c.freq[i] for i in range(c.tune_count)], c)


FNV_OFFSET = 14695981039346656037


def fnv1a_int64(words, h=FNV_OFFSET):
    """FNV-1a over int64 words in natural (hop-major) order: the hash of SURVEY.md 8(c)'s known-answer rows"""
    import numpy as np
    a = np.ascontiguousarray(words, dtype=np.int64)
    return int(host_library().synth_fnv1a_int64(a.ctypes.data, a.size, ctypes.c_uint64(h)))


def synth_cube(out_ptr, mode, seed, param, tune_count, hop_first, hop_count, pass_first, passes, buf_len,
               pass_stride=None, hop_stride=None, threads=None):
    """Fill [passes, hop_count, buf_len] (or the given strides) at out_ptr with the synthetic source's bytes
    for reads (pass_first + p, hop_first + k): a pure function of (mode, seed, hop, pass)."""
    hop_stride = buf_len if hop_stride is None else hop_stride
    pass_stride = hop_count * hop_stride if pass_stride is None else pass_stride
    threads = threads or min(32, os.cpu_count() or 1)
    host_library().synth_generate_cube(mode, ctypes.c_uint64(seed), param, tune_count, hop_first, hop_count,
                                       ctypes.c_uint64(pass_first), ctypes.c_uint64(passes), out_ptr,
                                       pass_stride, hop_stride, buf_len, threads)
