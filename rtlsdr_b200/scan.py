"""ctypes binding of include/rtlsdr_gpu_scan.h (the C ABI is the product boundary)."""
import ctypes
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class ScanError(RuntimeError):
    def __init__(self, code, what, detail=""):
        self.code = code
        super().__init__(f"{what}: error {code}" + (f" ({detail})" if detail else ""))


class _Cfg(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32), ("device", ctypes.c_int32),
                ("tune_count", ctypes.c_int32), ("bin_e", ctypes.c_int32),
                ("buf_len", ctypes.c_int32), ("downsample", ctypes.c_int32),
                ("downsample_passes", ctypes.c_int32), ("boxcar", ctypes.c_int32),
                ("comp_fir_size", ctypes.c_int32), ("peak_hold", ctypes.c_int32),
                ("rate", ctypes.c_int32), ("crop", ctypes.c_double),
                ("window_coefs", ctypes.c_void_p), ("sinewave", ctypes.c_void_p),
                ("ring_bytes", ctypes.c_uint32), ("flags", ctypes.c_uint32), ("iir_alpha", ctypes.c_double)]


def lib_path():
    """RTLSDR_GPU_SCAN_LIB selects another build of the same CUDA library (kernel experiments)."""
    return os.environ.get("RTLSDR_GPU_SCAN_LIB") or os.path.join(PKG, "librtlsdr_gpu_scan.so")


def load_library():
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise ScanError(-5, "librtlsdr_gpu_scan.so missing",
                        "run __graft_entry__.build() / rtlsdr_b200._build.build_cuda()")
    L = ctypes.CDLL(path)
    vp, i, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    L.rtlsdr_gpu_scan_init.argtypes = [ctypes.POINTER(_Cfg), ctypes.POINTER(vp)]
    L.rtlsdr_gpu_scan_close.argtypes = [vp]
    L.rtlsdr_gpu_scan_close.restype = None
    L.rtlsdr_gpu_scan_submit.argtypes = [vp, i, vp, ctypes.c_uint32]
    L.rtlsdr_gpu_scan_submit_batch.argtypes = [vp, i, i, i, vp, i64, i64]
    L.rtlsdr_gpu_scan_submit_device.argtypes = [vp, i, i, i, vp, i64, i64]
    L.rtlsdr_gpu_scan_submit_reads.argtypes = [vp, i, vp, vp, i64]
    L.rtlsdr_gpu_scan_flag_signal.argtypes = [vp, vp, ctypes.c_uint32]
    L.rtlsdr_gpu_scan_flag_signal_many.argtypes = [vp, vp, i, ctypes.c_uint32]
    L.rtlsdr_gpu_scan_flag_wait.argtypes = [vp, vp, i, ctypes.c_uint32, ctypes.c_uint32, vp]
    L.rtlsdr_gpu_scan_flush.argtypes = [vp]
    L.rtlsdr_gpu_scan_sync.argtypes = [vp]
    L.rtlsdr_gpu_scan_collect.argtypes = [vp, i, vp, vp, vp]
    L.rtlsdr_gpu_scan_collect_all.argtypes = [vp, vp, vp, vp]
    L.rtlsdr_gpu_scan_collect_device.argtypes = [vp, vp, vp, vp]
    L.rtlsdr_gpu_scan_collect_sk.argtypes = [vp, vp, vp, vp, vp, vp]
    L.rtlsdr_gpu_scan_merge_device.argtypes = [vp, vp, vp, i, i64]
    L.rtlsdr_gpu_scan_collect_sk_device.argtypes = [vp, vp, vp, vp, vp, vp]
    L.rtlsdr_gpu_scan_merge_sk_device.argtypes = [vp, vp, vp, vp, i, i64]
    L.rtlsdr_gpu_scan_sk_csv_capacity.argtypes = [vp, i, ctypes.c_size_t]
    L.rtlsdr_gpu_scan_sk_csv_capacity.restype = i64
    L.rtlsdr_gpu_scan_format_sk_csv_device.argtypes = [vp, ctypes.c_char_p, i, i, vp, i64, vp, vp, ctypes.c_size_t, vp]
    L.rtlsdr_gpu_scan_collect_sk_csv.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_size_t,
                                                 ctypes.POINTER(ctypes.c_size_t), vp, ctypes.c_size_t,
                                                 ctypes.POINTER(ctypes.c_size_t)]
    L.rtlsdr_gpu_scan_set_csv_columns.argtypes = [vp, i, vp, vp, ctypes.c_double]
    L.rtlsdr_gpu_scan_csv_capacity.argtypes = [vp, i, ctypes.c_size_t]
    L.rtlsdr_gpu_scan_csv_capacity.restype = i64
    L.rtlsdr_gpu_scan_collect_csv.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    L.rtlsdr_gpu_scan_format_csv_device.argtypes = [vp, ctypes.c_char_p, i, i, vp, i64, vp, vp, ctypes.c_size_t, vp]
    L.rtlsdr_gpu_scan_db_count.argtypes = [vp]
    L.rtlsdr_gpu_scan_host_alloc.argtypes = [ctypes.c_size_t]
    L.rtlsdr_gpu_scan_host_alloc.restype = vp
    L.rtlsdr_gpu_scan_host_free.argtypes = [vp]
    L.rtlsdr_gpu_scan_host_free.restype = None
    L.rtlsdr_gpu_scan_set_stream.argtypes = [vp, vp]
    L.rtlsdr_gpu_scan_get_stream.argtypes = [vp]
    L.rtlsdr_gpu_scan_get_stream.restype = vp
    L.rtlsdr_gpu_scan_get_report_stream.argtypes = [vp]
    L.rtlsdr_gpu_scan_get_report_stream.restype = vp
    L.rtlsdr_gpu_scan_sine_table.argtypes = [i, vp]
    L.rtlsdr_gpu_scan_sine_table.restype = None
    L.rtlsdr_gpu_scan_window.argtypes = [ctypes.c_char_p, i, vp]
    L.rtlsdr_gpu_scan_stats.argtypes = [vp, vp, vp, vp]
    L.rtlsdr_gpu_scan_level_stats.argtypes = [vp, i, vp, vp, vp]
    L.rtlsdr_gpu_scan_kernel_time.argtypes = [vp, vp, vp]
    L.rtlsdr_gpu_scan_set_timing.argtypes = [vp, i]
    L.rtlsdr_gpu_scan_strerror.argtypes = [i]
    L.rtlsdr_gpu_scan_strerror.restype = ctypes.c_char_p
    L.rtlsdr_gpu_scan_last_cuda_error.argtypes = [vp]
    L.rtlsdr_gpu_scan_last_cuda_error.restype = ctypes.c_char_p
    _LIB = L
    return L


def window_coefs(name, n):
    """window_coefs[] for a -w name, built on the host like rtl_power.c:985-988."""
    out = np.zeros(n, dtype=np.int32)
    load_library().rtlsdr_gpu_scan_window(name.encode(), n, out.ctypes.data_as(ctypes.c_void_p))
    return out


def sine_table(bin_e):
    out = np.zeros(max((1 << bin_e) * 3 // 4, 1), dtype=np.int16)
    load_library().rtlsdr_gpu_scan_sine_table(bin_e, out.ctypes.data_as(ctypes.c_void_p))
    return out[: (1 << bin_e) * 3 // 4]


def flag_signal(cuda_stream, dev_flag, value):
    """one-thread kernel on `cuda_stream`: *dev_flag = value with system-scope release (may be peer memory)"""
    rc = load_library().rtlsdr_gpu_scan_flag_signal(cuda_stream, dev_flag, value & 0xFFFFFFFF)
    if rc:
        raise ScanError(rc, "flag_signal")


def flag_signal_many(cuda_stream, dev_flag_addrs, value):
    """one launch raising the flags at all the given device addresses (<= 32)"""
    arr = (ctypes.c_void_p * len(dev_flag_addrs))(*dev_flag_addrs)
    rc = load_library().rtlsdr_gpu_scan_flag_signal_many(cuda_stream, arr, len(dev_flag_addrs), value & 0xFFFFFFFF)
    if rc:
        raise ScanError(rc, "flag_signal_many")


def flag_wait(cuda_stream, dev_flags, count, value, timeout_ms=0, dev_timed_out=None):
    """kernel on `cuda_stream` that sleeps until dev_flags[0..count) have all reached `value`"""
    rc = load_library().rtlsdr_gpu_scan_flag_wait(cuda_stream, dev_flags, count, value & 0xFFFFFFFF, timeout_ms, dev_timed_out)
    if rc:
        raise ScanError(rc, "flag_wait")


class PinnedBuffer:
    """uint8 numpy view over memory from rtlsdr_gpu_scan_host_alloc()."""

    def __init__(self, nbytes):
        self._lib = load_library()
        self.ptr = self._lib.rtlsdr_gpu_scan_host_alloc(nbytes)
        if not self.ptr:
            raise ScanError(-7, "rtlsdr_gpu_scan_host_alloc")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(self.ptr))

    def view(self, dtype, shape, offset=0):
        """typed numpy view of a slice of the pinned block"""
        count = int(np.prod(shape))
        nbytes = count * np.dtype(dtype).itemsize
        return self.array[offset: offset + nbytes].view(dtype).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            self._lib.rtlsdr_gpu_scan_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class GpuScan:
    """One rtlsdr_gpu_scan_t handle.  Argument names are the reference's
    (tunes[0].bin_e, buf_len, downsample, ... see include/rtlsdr_gpu_scan.h)."""

    def __init__(self, tune_count, bin_e, buf_len, downsample=1, downsample_passes=0, boxcar=1,
                 comp_fir_size=0, peak_hold=0, rate=2400000, crop=0.0, window_coefs=None,
                 sinewave=None, device=0, ring_bytes=0, level_stats=False, iir_alpha=0.0, async_report=False,
                 short_reads=False, spectral_kurtosis=False):
        self.lib = load_library()
        self.tune_count, self.bin_e, self.buf_len = tune_count, bin_e, buf_len
        self.n = 1 << bin_e
        cfg = _Cfg()
        cfg.struct_size = ctypes.sizeof(_Cfg)
        cfg.device = device
        cfg.tune_count, cfg.bin_e, cfg.buf_len = tune_count, bin_e, buf_len
        cfg.downsample, cfg.downsample_passes = downsample, downsample_passes
        cfg.boxcar, cfg.comp_fir_size, cfg.peak_hold = boxcar, comp_fir_size, peak_hold
        cfg.rate, cfg.crop = rate, crop
        self._w = self._s = None
        if window_coefs is not None:
            self._w = np.ascontiguousarray(window_coefs, dtype=np.int32)
            assert self._w.size == self.n
            cfg.window_coefs = self._w.ctypes.data
        if sinewave is not None:
            self._s = np.ascontiguousarray(sinewave, dtype=np.int16)
            cfg.sinewave = self._s.ctypes.data
        cfg.ring_bytes = ring_bytes
        # RTLSDR_GPU_FLAG_LEVEL_STATS / _ASYNC_REPORT / _SHORT_READS / _SPECTRAL_KURTOSIS
        cfg.flags = ((1 if level_stats else 0) | (2 if async_report else 0) | (4 if short_reads else 0)
                     | (8 if spectral_kurtosis else 0))
        cfg.iir_alpha = iir_alpha            # -s iir smoothing of the dB rows across reports (0 = off)
        self.h = ctypes.c_void_p()
        rc = self.lib.rtlsdr_gpu_scan_init(ctypes.byref(cfg), ctypes.byref(self.h))
        if rc:
            self.h = None
            raise ScanError(rc, "rtlsdr_gpu_scan_init", self.lib.rtlsdr_gpu_scan_strerror(rc).decode())
        self.db_count = self.lib.rtlsdr_gpu_scan_db_count(self.h)

    @classmethod
    def from_plan(cls, plan, window_coefs=None, peak_hold=0, device=0, hops=None, **kw):
        """plan: rtlsdr_b200.planner.Plan or the dict tests get from the oracle."""
        g = plan if isinstance(plan, dict) else plan.as_dict()
        tc = g["tune_count"] if hops is None else len(hops)
        return cls(tc, g["bin_e"], g["buf_len"], g["downsample"], g["downsample_passes"],
                   g["boxcar"], g["comp_fir_size"], g.get("peak_hold", peak_hold), g["rate"],
                   g["crop"], window_coefs, device=device, **kw)

    def _check(self, rc, what):
        if rc:
            detail = self.lib.rtlsdr_gpu_scan_strerror(rc).decode()
            cu = self.lib.rtlsdr_gpu_scan_last_cuda_error(self.h).decode() if self.h else ""
            raise ScanError(rc, what, detail + ("; " + cu if cu else ""))

    def submit(self, hop, buf):
        b = np.ascontiguousarray(buf, dtype=np.uint8)
        self._check(self.lib.rtlsdr_gpu_scan_submit(self.h, hop, b.ctypes.data, b.size), "submit")

    def submit_batch(self, hop_first, hop_count, passes, host_ptr, pass_stride, hop_stride):
        self._check(self.lib.rtlsdr_gpu_scan_submit_batch(self.h, hop_first, hop_count, passes, host_ptr,
                                                          pass_stride, hop_stride), "submit_batch")

    def submit_reads(self, hops, host_ptr, stride=None):
        """hop visits in any order: read i (buf_len bytes at host_ptr + i * stride, pinned memory) belongs to hops[i]"""
        hp = np.ascontiguousarray(hops, dtype=np.int32)
        self._check(self.lib.rtlsdr_gpu_scan_submit_reads(self.h, hp.size, hp.ctypes.data, host_ptr,
                                                          self.buf_len if stride is None else stride), "submit_reads")

    def submit_device(self, hop_first, hop_count, passes, dev_ptr, pass_stride, hop_stride):
        self._check(self.lib.rtlsdr_gpu_scan_submit_device(self.h, hop_first, hop_count, passes, dev_ptr,
                                                           pass_stride, hop_stride), "submit_device")

    def flush(self):
        self._check(self.lib.rtlsdr_gpu_scan_flush(self.h), "flush")

    def sync(self):
        self._check(self.lib.rtlsdr_gpu_scan_sync(self.h), "sync")

    def collect(self, hop, want_db=True):
        avg = np.zeros(self.n, dtype=np.int64)
        db = np.zeros(self.db_count, dtype=np.float64) if want_db else None
        smp = ctypes.c_int(0)
        self._check(self.lib.rtlsdr_gpu_scan_collect(self.h, hop, avg.ctypes.data, ctypes.byref(smp),
                                                     db.ctypes.data if want_db else None), "collect")
        return avg, smp.value, db

    def collect_all(self, want_db=True, out=None):
        """out: optional (avg int64 [tc, N], samples int32 [tc], db float64 [tc, db_count]) arrays to
        fill, e.g. views of pinned memory (PinnedBuffer) so the device-to-host copies are asynchronous."""
        if out is not None:
            avg, smp, db = out
        else:
            avg = np.zeros((self.tune_count, self.n), dtype=np.int64)
            smp = np.zeros(self.tune_count, dtype=np.int32)
            db = np.zeros((self.tune_count, self.db_count), dtype=np.float64) if want_db else None
        self._check(self.lib.rtlsdr_gpu_scan_collect_all(self.h, avg.ctypes.data, smp.ctypes.data,
                                                         db.ctypes.data if db is not None else None), "collect_all")
        return avg, smp, db

    def collect_sk(self):
        """collect_all() plus the spectral-kurtosis report (spectral_kurtosis=True handles):
        (avg int64 [tc, N], samples int32 [tc], db float64 [tc, db_count],
         s2 uint64 [tc, N, 2] the 128-bit sums of |X|^4 as (lo, hi), sk float64 [tc, db_count] in the dB row's layout)"""
        avg = np.zeros((self.tune_count, self.n), dtype=np.int64)
        smp = np.zeros(self.tune_count, dtype=np.int32)
        db = np.zeros((self.tune_count, self.db_count), dtype=np.float64)
        s2 = np.zeros((self.tune_count, self.n, 2), dtype=np.uint64)
        sk = np.zeros((self.tune_count, self.db_count), dtype=np.float64)
        self._check(self.lib.rtlsdr_gpu_scan_collect_sk(self.h, avg.ctypes.data, smp.ctypes.data, db.ctypes.data,
                                                        s2.ctypes.data, sk.ctypes.data), "collect_sk")
        return avg, smp, db, s2, sk

    def collect_device(self, dev_avg=None, dev_samples=None, dev_db=None):
        self._check(self.lib.rtlsdr_gpu_scan_collect_device(self.h, dev_avg, dev_samples, dev_db), "collect_device")

    def merge_device(self, dev_avg, dev_samples, sets=1, set_stride=0):
        """fold `sets` external accumulator sets (raw int64 bins + int32 counts as collect_device writes them,
        `set_stride` bytes apart; may be peer memory) into this handle's: sums, or maxima under peak hold"""
        self._check(self.lib.rtlsdr_gpu_scan_merge_device(self.h, dev_avg, dev_samples, sets, set_stride), "merge_device")

    def collect_sk_device(self, dev_avg=None, dev_samples=None, dev_db=None, dev_s2=None, dev_sk=None):
        """collect_device() plus S2 (uint64 [tc, N, 2]) and the SK rows (float64 [tc, db_count]) of a
        spectral_kurtosis=True handle; any address may be None; async on the handle's stream"""
        self._check(self.lib.rtlsdr_gpu_scan_collect_sk_device(self.h, dev_avg, dev_samples, dev_db, dev_s2, dev_sk),
                    "collect_sk_device")

    def merge_sk_device(self, dev_avg, dev_samples, dev_s2, sets=1, set_stride=0):
        """merge_device() plus S2 (what collect_sk_device wrote, `set_stride` bytes apart like the other two),
        added as exact 128-bit sums"""
        self._check(self.lib.rtlsdr_gpu_scan_merge_sk_device(self.h, dev_avg, dev_samples, dev_s2, sets, set_stride),
                    "merge_sk_device")

    def set_csv_columns(self, low, high, step):
        """row table of the CSV formatter: row r prints low[r], high[r], step (Plan.csv_columns())"""
        lo = np.ascontiguousarray(low, dtype=np.int32)
        hi = np.ascontiguousarray(high, dtype=np.int32)
        assert lo.size == hi.size
        self._check(self.lib.rtlsdr_gpu_scan_set_csv_columns(self.h, lo.size, lo.ctypes.data, hi.ctypes.data,
                                                             float(step)), "set_csv_columns")

    def csv_capacity(self, rows, stamp_len):
        """bytes `rows` CSV rows with a stamp of `stamp_len` bytes can take at most"""
        n = self.lib.rtlsdr_gpu_scan_csv_capacity(self.h, rows, stamp_len)
        self._check(n if n < 0 else 0, "csv_capacity")
        return n

    def collect_csv(self, stamp, out=None):
        """collect_all()'s read-and-zero, returning the rows' text (bytes), formatted on the GPU.  `stamp` is
        printed verbatim before every row; out: optional writable uint8 buffer (e.g. PinnedBuffer.array)."""
        s = stamp.encode() if isinstance(stamp, str) else bytes(stamp)
        if out is None:
            out = np.empty(max(1, self.csv_capacity(self.tune_count, len(s))), dtype=np.uint8)
        n = ctypes.c_size_t(0)
        self._check(self.lib.rtlsdr_gpu_scan_collect_csv(self.h, s, out.ctypes.data, out.nbytes, ctypes.byref(n)),
                    "collect_csv")
        return out[: n.value].tobytes()

    def sk_csv_capacity(self, rows, stamp_len):
        """bytes `rows` spectral-kurtosis rows with a stamp of `stamp_len` bytes can take at most"""
        n = self.lib.rtlsdr_gpu_scan_sk_csv_capacity(self.h, rows, stamp_len)
        self._check(n if n < 0 else 0, "sk_csv_capacity")
        return n

    def collect_sk_csv(self, stamp, out=None, sk_out=None):
        """collect_csv() plus the spectral-kurtosis rows: (power rows' text, SK rows' text) as bytes, formatted on
        the GPU; out / sk_out: optional writable uint8 buffers"""
        s = stamp.encode() if isinstance(stamp, str) else bytes(stamp)
        if out is None:
            out = np.empty(max(1, self.csv_capacity(self.tune_count, len(s))), dtype=np.uint8)
        if sk_out is None:
            sk_out = np.empty(max(1, self.sk_csv_capacity(self.tune_count, len(s))), dtype=np.uint8)
        n, m = ctypes.c_size_t(0), ctypes.c_size_t(0)
        self._check(self.lib.rtlsdr_gpu_scan_collect_sk_csv(self.h, s, out.ctypes.data, out.nbytes, ctypes.byref(n),
                                                            sk_out.ctypes.data, sk_out.nbytes, ctypes.byref(m)),
                    "collect_sk_csv")
        return out[: n.value].tobytes(), sk_out[: m.value].tobytes()

    def format_sk_csv_device(self, stamp, row_first, rows, dev_sk, sk_stride, dev_samples, dev_text, cap, dev_len):
        """format_csv_device() for the SK rows of a collect_sk_device() report (sk_stride doubles apart)"""
        s = stamp.encode() if isinstance(stamp, str) else bytes(stamp)
        self._check(self.lib.rtlsdr_gpu_scan_format_sk_csv_device(self.h, s, row_first, rows, dev_sk, sk_stride,
                                                                  dev_samples, dev_text, cap, dev_len),
                    "format_sk_csv_device")

    def format_csv_device(self, stamp, row_first, rows, dev_db, db_stride, dev_samples, dev_text, cap, dev_len):
        """rows [row_first, row_first + rows) of a collect_device() report (dB rows db_stride doubles apart,
        int32 counts) into dev_text / *dev_len (int64, -1 = value outside the domain), async on the handle's stream"""
        s = stamp.encode() if isinstance(stamp, str) else bytes(stamp)
        self._check(self.lib.rtlsdr_gpu_scan_format_csv_device(self.h, s, row_first, rows, dev_db, db_stride,
                                                               dev_samples, dev_text, cap, dev_len),
                    "format_csv_device")

    def set_stream(self, cuda_stream):
        self._check(self.lib.rtlsdr_gpu_scan_set_stream(self.h, cuda_stream), "set_stream")

    def level_stats(self, hop):
        """(overload, high_level, bytes) soft-AGC byte counts of `hop` since its last collect"""
        a, b, c = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self.lib.rtlsdr_gpu_scan_level_stats(self.h, hop, ctypes.byref(a), ctypes.byref(b),
                                                         ctypes.byref(c)), "level_stats")
        return a.value, b.value, c.value

    def get_stream(self):
        """raw cudaStream_t of the handle (wrap with torch.cuda.ExternalStream to record events on it)"""
        return self.lib.rtlsdr_gpu_scan_get_stream(self.h)

    def get_report_stream(self):
        """raw cudaStream_t collect_device() reports on (the handle's stream unless async_report=True)"""
        return self.lib.rtlsdr_gpu_scan_get_report_stream(self.h)

    def stats(self):
        k, a, b = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        self.lib.rtlsdr_gpu_scan_stats(self.h, ctypes.byref(k), ctypes.byref(a), ctypes.byref(b))
        return dict(kernel_launches=k.value, h2d_bytes=a.value, d2h_bytes=b.value)

    def set_timing(self, every):
        """bracket every `every`-th transform kernel with CUDA events (0 = off)"""
        self._check(self.lib.rtlsdr_gpu_scan_set_timing(self.h, every), "set_timing")

    def kernel_time(self):
        """(ms, launches) of the transform kernels since the previous call; the first call arms timing."""
        ms, n = ctypes.c_double(), ctypes.c_uint64()
        self._check(self.lib.rtlsdr_gpu_scan_kernel_time(self.h, ctypes.byref(ms), ctypes.byref(n)), "kernel_time")
        return ms.value, n.value

    def close(self):
        if self.h:
            self.lib.rtlsdr_gpu_scan_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
