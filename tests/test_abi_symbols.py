"""The C-ABI library builds for sm_100a, loads, and exports exactly what
include/rtlsdr_gpu_scan.h declares.  No compute calls: there is no GPU here."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rtlsdr_gpu_scan.h")


@pytest.fixture(scope="module")
def lib():
    from rtlsdr_b200 import _build
    import rtlsdr_b200.scan as rs
    _build.build_cuda()
    return rs.load_library()


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"RTLSDR_GPU_API[^;(]*?\b(rtlsdr_gpu_scan_\w+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
    # and nothing else leaks out of the library (hidden default visibility, like CMakeLists.txt:54)
    from rtlsdr_b200.scan import lib_path
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path()], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert exported == set(names), exported ^ set(names)


def test_library_contains_sm100a_code_only():
    from rtlsdr_b200.scan import lib_path
    out = subprocess.run(["cuobjdump", "-lelf", lib_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert not re.search(r"sm_(?!100a)\d+", out), out


def test_null_and_config_errors_without_gpu(lib):
    h = ctypes.c_void_p()
    assert lib.rtlsdr_gpu_scan_init(None, ctypes.byref(h)) == -1
    assert lib.rtlsdr_gpu_scan_submit(None, 0, None, 0) == -1
    assert lib.rtlsdr_gpu_scan_collect(None, 0, None, None, None) == -1
    assert lib.rtlsdr_gpu_scan_flush(None) == -1
    assert lib.rtlsdr_gpu_scan_db_count(None) == -1
    assert lib.rtlsdr_gpu_scan_strerror(-3) == b"hop index out of range"
    lib.rtlsdr_gpu_scan_close(None)  # no-op like free(NULL)


def test_no_cpu_fallback(lib):
    """Without a usable sm_100 device init must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import rtlsdr_b200.scan as rs
    with pytest.raises(rs.ScanError) as e:
        rs.GpuScan(1, 10, 16384)
    assert e.value.code in (-5, -6)


def test_host_table_helpers_match_oracle(lib, port_oracle):
    import rtlsdr_b200.scan as rs
    from oracles import WINDOWS
    for m in (1, 2, 5, 10, 13):
        assert np.array_equal(rs.sine_table(m), port_oracle.sine_table(m))
    for w in WINDOWS:
        for n in (2, 64, 4096):
            assert np.array_equal(rs.window_coefs(w, n), port_oracle.window_coefs(w, n)), (w, n)
    out = np.zeros(8, dtype=np.int32)
    assert lib.rtlsdr_gpu_scan_window(b"nonsense", 8, out.ctypes.data_as(ctypes.c_void_p)) == -1
    assert (out == 256).all()  # unknown names silently stay rectangle (rtl_power.c:826-843)


def test_config_validation_happens_before_any_device_work(lib):
    """malformed configurations are rejected with RTLSDR_GPU_ERR_CONFIG (-2) even without a GPU"""
    import rtlsdr_b200.scan as rs

    def init(**kw):
        cfg = rs._Cfg()
        cfg.struct_size = ctypes.sizeof(rs._Cfg)
        base = dict(device=0, tune_count=1, bin_e=10, buf_len=16384, downsample=1, downsample_passes=0,
                    boxcar=1, comp_fir_size=0, peak_hold=0, rate=2400000, crop=0.0)
        base.update(kw)
        for k, v in base.items():
            setattr(cfg, k, v)
        h = ctypes.c_void_p()
        return lib.rtlsdr_gpu_scan_init(ctypes.byref(cfg), ctypes.byref(h))

    assert init(struct_size=8) == -2                 # ABI version mismatch
    assert init(tune_count=0) == -2
    assert init(tune_count=3001) == -2               # MAX_TUNES, rtl_power.c:113
    assert init(bin_e=22) == -2                      # planner stops at 21, rtl_power.c:483
    assert init(buf_len=1000) == -2                  # not a multiple of 16
    assert init(rate=0) == -2
    assert init(crop=1.5) == -2
    assert init(downsample=0) == -2
    assert init(boxcar=0, downsample=8, downsample_passes=2) == -2   # ds must be 2^passes with -F
    assert init(boxcar=0, downsample=3, downsample_passes=0) == -2   # ds > 1 without a decimator
    assert init(bin_e=10, buf_len=32768) == -2       # u8 path: the planner's 16384-byte reads only
    assert init(bin_e=14, buf_len=16384) == -2       # large path: exactly one FFT block per read
    assert init(bin_e=1, crop=1.0) == -2             # the crop leaves no bin printed
    sine = rs.sine_table(10)
    sine[0] = 1                                      # the kernels need Sinewave[0] = Sinewave[N/2] = 0
    assert init(sinewave=sine.ctypes.data) == -2
