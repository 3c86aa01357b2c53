"""Spectral kurtosis (RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS) without a GPU: the oracle's S2, sk.cuh's 128-bit
conversion and estimator against gcc and Python doubles, and the SK kernels run through the CPU emulator
(tests/emu/sk_entry.cpp) against the oracle, exactly."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracles import SYNTH_BIASED, SYNTH_XORSHIFT, OracleCfg, _ptr
from scan_cases import make_reads, plan_dict
from test_emu_kernels import emu, sort_by_hop, vp  # noqa: F401  (emu: fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")
SK_SO = os.path.join(EMU_DIR, "libsk_emu.so")
ORACLE_SK_SO = os.path.join(ROOT, "tests", "liboracle_sk.so")
U64 = (1 << 64) - 1
_oracle_sk_lib = None


def oracle_sk_lib():
    """tests/oracle_sk.c: oracle_scan_read_sk, built with the oracle's flags"""
    global _oracle_sk_lib
    if _oracle_sk_lib is None:
        src = os.path.join(ROOT, "tests", "oracle_sk.c")
        deps = [src] + [os.path.join(ROOT, "oracle", f) for f in ("scan_oracle.c", "scan_oracle.h")]
        if not os.path.exists(ORACLE_SK_SO) or any(os.path.getmtime(d) > os.path.getmtime(ORACLE_SK_SO) for d in deps):
            subprocess.run(["gcc", "-O3", "-DNDEBUG", "-fwrapv", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "oracle"),
                            "-o", ORACLE_SK_SO, src, "-lm"], check=True)
        _oracle_sk_lib = ctypes.CDLL(ORACLE_SK_SO)
        _oracle_sk_lib.oracle_scan_read_sk.argtypes = [ctypes.c_void_p] * 6
    return _oracle_sk_lib


def oracle_sk(port_oracle, plan, window, reads, hops):
    """PortOracle.scan() through oracle_scan_read_sk: (avg, samples, s2 uint64 [tune_count, N, 2] = (lo, hi) of
    the 128-bit sum of |X|^4).  Sums only, bin_e >= 1."""
    lib = oracle_sk_lib()
    n, tc = 1 << plan["bin_e"], plan["tune_count"]
    sine = np.ascontiguousarray(np.concatenate([port_oracle.sine_table(plan["bin_e"]), np.zeros(4, np.int16)]))
    window = np.ascontiguousarray(window, dtype=np.int32)
    cfg = OracleCfg(plan["bin_e"], plan["buf_len"], plan["downsample"], plan["downsample_passes"], plan["boxcar"],
                    plan["comp_fir_size"], 0, window.ctypes.data, sine.ctypes.data)
    avg = np.zeros((tc, n), dtype=np.int64)
    samples = np.zeros(tc, dtype=np.int32)
    s2 = np.zeros((tc, n, 2), dtype=np.uint64)
    work = np.zeros(plan["buf_len"] + 16, dtype=np.int16)
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    for i, h in enumerate(hops):
        s = ctypes.c_int(int(samples[h]))
        lib.oracle_scan_read_sk(ctypes.addressof(cfg), _ptr(reads[i]), _ptr(work), _ptr(avg[h]), ctypes.addressof(s),
                                _ptr(s2[h]))
        samples[h] = s.value
    return avg, samples, s2


@pytest.fixture(scope="module")
def sk_emu():
    srcs = [os.path.join(EMU_DIR, f) for f in ("sk_entry.cpp", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".inl"))]
    srcs.append(os.path.join(ROOT, "include", "rtlsdr_gpu_scan.h"))
    if not os.path.exists(SK_SO) or any(os.path.getmtime(s) > os.path.getmtime(SK_SO) for s in srcs):
        subprocess.run(["g++", "-std=c++20", "-O2", "-ffp-contract=off", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC,
                        "-shared", "-fPIC", "-pthread", "-o", SK_SO, os.path.join(EMU_DIR, "sk_entry.cpp")], check=True)
    L = ctypes.CDLL(SK_SO)
    u64, i64 = ctypes.c_uint64, ctypes.c_int64
    for f in ("emu_sk_u128_to_double", "emu_gcc_u128_to_double"):
        getattr(L, f).argtypes = [u64, u64]
        getattr(L, f).restype = ctypes.c_double
    L.emu_sk_from_moments.argtypes = [i64, u64, u64, i64]
    L.emu_sk_from_moments.restype = ctypes.c_double
    return L


def s2_int(s2):
    """uint64 [..., 2] (lo, hi) -> Python ints"""
    s2 = np.asarray(s2, dtype=np.uint64)
    return [int(lo) | (int(hi) << 64) for lo, hi in s2.reshape(-1, 2)]


def sk_py(S1, S2, M):
    """the header's evaluation order in Python doubles (correctly rounded int -> float, IEEE operations)"""
    if M < 2 or S1 == 0:
        return float("nan")
    s1, s2 = float(S1), float(S2)
    a = float(M) * s2
    b = s1 * s1
    d = a / b - 1.0
    return (float(M + 1) / float(M - 1)) * d


def same_bits(a, b):
    return np.float64(a).tobytes() == np.float64(b).tobytes() or (a != a and b != b)


# ---- sk.cuh on the host ---------------------------------------------------------------------------------

def u128_patterns():
    rng = np.random.default_rng(7)
    vals = [0, 1, U64, U64 + 1, (1 << 128) - 1, 1 << 127]
    for k in range(0, 75):
        for base in ((1 << 53) - 1, 1 << 53, (1 << 53) + 1, (1 << 53) + 2, (1 << 54) - 1, (1 << 53) + 3):
            v = base << k
            vals += [v, v + 1, v - 1 if v else 0]
        # exact ties at every position of the low word, with and without a sticky bit below
        t = ((1 << 53) + 1) << (k + 1) | (1 << k)
        vals += [t, t + 1, t - 1]
    for _ in range(20000):
        bits = int(rng.integers(1, 129))
        vals.append(int.from_bytes(rng.bytes(16), "little") & ((1 << bits) - 1))
    return [v for v in vals if 0 <= v < (1 << 128)]


def test_u128_to_double_matches_gcc(sk_emu):
    bad = []
    for v in u128_patterns():
        got = sk_emu.emu_sk_u128_to_double(v & U64, v >> 64)
        want = sk_emu.emu_gcc_u128_to_double(v & U64, v >> 64)
        if not same_bits(got, want) or got != float(v):
            bad.append(v)
    assert not bad, [hex(v) for v in bad[:5]]


def test_sk_from_moments_matches_plain_evaluation(sk_emu):
    rng = np.random.default_rng(11)
    cases = [(0, 5, 10), (1, 0, 1), (1, 1, 0), (12345, 99, 1), (4, 16, 2), (1 << 62, 1 << 127, 2),
             ((1 << 63) - 1, (1 << 128) - 1, 1 << 40)]
    for _ in range(20000):
        m = int(rng.integers(0, 1 << int(rng.integers(1, 31))))
        s1 = int(rng.integers(0, 1 << 62))
        s2 = int.from_bytes(rng.bytes(16), "little") >> int(rng.integers(0, 128))
        cases.append((s1, s2, m))
    for s1, s2, m in cases:
        got = sk_emu.emu_sk_from_moments(s1, s2 & U64, s2 >> 64, m)
        assert same_bits(got, sk_py(s1, s2, m)), (s1, s2, m)
    assert np.isnan(sk_emu.emu_sk_from_moments(0, 5, 0, 10))   # S1 = 0
    assert np.isnan(sk_emu.emu_sk_from_moments(7, 49, 0, 1))   # M < 2


# ---- oracle -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("bin_e", [4, 10])
def test_oracle_s2_is_the_sum_of_squared_block_powers(port_oracle, bin_e):
    n = 1 << bin_e
    plan = plan_dict(bin_e, tune_count=1)
    win = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=bin_e, param=30)
    avg, smp, s2 = oracle_sk(port_oracle, plan, win, reads, hops)
    want_avg, want_smp = port_oracle.scan(plan, win, reads, hops, 1)
    assert np.array_equal(avg, want_avg) and np.array_equal(smp, want_smp)
    sine = port_oracle.sine_table(bin_e)
    tot = [0] * n
    for r in reads:
        work = (r.astype(np.int32) - 127).astype(np.int16)
        work = port_oracle.remove_dc(work, len(work))
        work[1:] = port_oracle.remove_dc(work[1:], len(work) - 1)
        for off in range(0, len(work), 2 * n):
            blk = work[off:off + 2 * n].astype(np.int32).reshape(n, 2) * win[:, None].astype(np.int32)
            blk = port_oracle.fix_fft(blk.astype(np.int16).reshape(-1), bin_e, sine)
            for j in range(n):
                p = int(blk[2 * j]) ** 2 + int(blk[2 * j + 1]) ** 2
                tot[j] += p * p
    assert s2_int(s2[0]) == tot


# ---- the SK kernels through the emulator --------------------------------------------------------------

def full_scale(buf_len):
    """0x00 / 0xFF in alternate samples: a full-scale tone whose pw^2 overflows 64 bits in four blocks"""
    b = np.zeros(buf_len, dtype=np.uint8)
    b[0::4] = b[1::4] = 255
    return b


@pytest.mark.parametrize("bin_e", [4, 10, 12])
def test_small_u8_sk_kernel(sk_emu, port_oracle, bin_e):
    n = 1 << bin_e
    plan = plan_dict(bin_e, tune_count=2)
    win = port_oracle.window_coefs("rectangle", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=10)
    reads[1::2] = full_scale(16384)    # every read of hop 1
    want_avg, want_smp, want_s2 = oracle_sk(port_oracle, plan, win, reads, hops)
    assert want_s2[..., 1].any(), "the full-scale reads must carry into the high word"
    sreads, shops, _ = sort_by_hop(reads, hops, 2)
    shops = np.ascontiguousarray(shops, dtype=np.int32)
    sine = port_oracle.sine_table(bin_e)
    for grid in (1, 4):
        avg = np.zeros((2, n), dtype=np.int64)
        smp = np.zeros(2, dtype=np.int64)
        s2 = np.zeros((2, n, 2), dtype=np.uint64)
        sk_emu.emu_sk_small_u8(bin_e, vp(sreads), len(sreads), vp(shops), grid, vp(sine), vp(win), vp(avg),
                               vp(smp), vp(s2))
        assert np.array_equal(avg, want_avg), grid
        assert np.array_equal(smp, want_smp), grid
        assert np.array_equal(s2, want_s2), grid


@pytest.mark.parametrize("freq,fir", [("100M:100.1M:100", -1), ("100M:100.3M:3k", 5)])
def test_small_in16_sk_kernel(emu, sk_emu, port_oracle, freq, fir):
    """decimated images: a narrow boxcar scan (ds = 28 at 1024 bins) and a -F 5 scan"""
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(freq, 0.0, None if fir < 0 else fir).as_dict()
    plan["peak_hold"] = 0
    bin_e, n = plan["bin_e"], 1 << plan["bin_e"]
    box = plan["boxcar"] and plan["downsample"] > 1
    assert box == (fir < 0)
    win = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_XORSHIFT, seed=5)
    reads[1] = full_scale(plan["buf_len"])
    want_avg, want_smp, want_s2 = oracle_sk(port_oracle, plan, win, reads, hops)
    sine = port_oracle.sine_table(bin_e)
    # the library's decimators write the images and DC sums (test_emu_kernels.py checks them), then the SK kernel
    l_len = plan["buf_len"] // plan["downsample"]
    blocks = (l_len + 2 * n - 1) // (2 * n)
    padded = blocks
    while (padded * n) % 4:
        padded += 1
    images = np.zeros((len(reads), padded * n), dtype=np.uint32)
    sums = np.zeros((len(reads), 2), dtype=np.int64)
    segs = np.array([(0, 0, len(reads), 0)], dtype=np.int32)
    scratch = np.zeros((1, n), dtype=np.int64)
    emu.emu_small_decim(bin_e, 0, vp(reads), len(reads), plan["buf_len"], plan["downsample"],
                        plan["downsample_passes"], 0 if box else 1, None, vp(segs), 1, vp(sine), vp(win),
                        vp(scratch), vp(images), vp(sums))
    for segs in (np.array([(0, 0, 3, 0)], dtype=np.int32), np.array([(0, 0, 1, 0), (0, 1, 2, 0)], dtype=np.int32)):
        avg = np.zeros((1, n), dtype=np.int64)
        smp = np.zeros(1, dtype=np.int64)
        s2 = np.zeros((1, n, 2), dtype=np.uint64)
        sk_emu.emu_sk_small_in16(bin_e, vp(images), vp(sums), len(reads), plan["buf_len"], plan["downsample"],
                                 plan["downsample_passes"], 1 if box else 0, vp(segs), len(segs), vp(sine), vp(win),
                                 vp(avg), vp(smp), vp(s2))
        assert np.array_equal(avg, want_avg), len(segs)
        assert np.array_equal(smp, want_smp), len(segs)
        assert np.array_equal(s2, want_s2), len(segs)


@pytest.mark.parametrize("bin_e", [13, 17])
def test_large_sk_kernels(sk_emu, port_oracle, bin_e):
    """round B (N <= 2^16) and round C (N >= 2^17) with S2; two hops, one of them with a full-scale read"""
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=2 * n, tune_count=2)
    win = port_oracle.window_coefs("rectangle", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=35)
    reads, hops = reads[:5], hops[:5]
    reads[2] = full_scale(2 * n)
    want_avg, _, want_s2 = oracle_sk(port_oracle, plan, win, reads, hops)
    sreads, shops, _ = sort_by_hop(reads, hops, 2)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((2, n), dtype=np.int64)
    s2 = np.zeros((2, n, 2), dtype=np.uint64)
    sk_emu.emu_sk_large(bin_e, vp(sreads), len(sreads), vp(shops.astype(np.int32)), vp(sine), vp(win), vp(avg), vp(s2))
    assert np.array_equal(avg, want_avg)
    assert np.array_equal(s2, want_s2)


def expected_sk_rows(avg, smp, s2, bin_e, crop, ds, f=sk_py):
    """the dB row's layout (rtl_power.c:732-760): bin 0 takes bin 1, half swap, crop [i1, i2], duplicate of i2"""
    n = 1 << bin_e
    i1, i2 = int(n * crop * 0.5), (n - 1) - int(n * crop * 0.5)
    rows = []
    for h in range(avg.shape[0]):
        S2 = s2_int(s2[h])
        row = []
        for i in list(range(i1, i2 + 1)) + [i2]:
            j = (i + n // 2) & (n - 1)
            j = 1 if j == 0 else j
            row.append(f(int(avg[h, j]), S2[j], int(smp[h]) // ds))
        rows.append(row)
    return np.array(rows), i1, i2


@pytest.mark.parametrize("bin_e,crop,ds", [(1, 0.0, 1), (5, 0.0, 1), (10, 0.3, 28)])
def test_sk_report_kernel_layout(sk_emu, bin_e, crop, ds):
    rng = np.random.default_rng(bin_e)
    n = 1 << bin_e
    avg = rng.integers(0, 1 << 50, (3, n)).astype(np.int64)
    avg[2, 3 % n] = 0
    s2 = rng.integers(0, 1 << 63, (3, n, 2), dtype=np.uint64)
    s2[0, :, 1] = 0
    smp = np.array([ds * 40, ds, 0], dtype=np.int64)   # M = 40, M = 1 (NaN row), M = 0 (NaN row)
    want, i1, i2 = expected_sk_rows(avg, smp, s2, bin_e, crop, ds)
    got = np.zeros_like(want)
    sk_emu.emu_sk_report(vp(avg), vp(smp), vp(s2), vp(got), bin_e, i1, i2, ds, 3)
    assert all(same_bits(a, b) for a, b in zip(got.ravel(), want.ravel()))
    assert np.isnan(got[1:]).all() and np.isfinite(got[0]).all()


def test_sk_config_errors_before_any_device_work():
    """SK with peak hold, with the rms path (bin_e 0) or with an asynchronous report: RTLSDR_GPU_ERR_CONFIG"""
    import rtlsdr_b200.scan as rs
    from rtlsdr_b200 import _build
    _build.build_cuda()
    for kw in (dict(bin_e=10, peak_hold=1), dict(bin_e=0), dict(bin_e=10, async_report=True)):
        bin_e = kw.pop("bin_e")
        with pytest.raises(rs.ScanError) as e:
            rs.GpuScan(2, bin_e, 16384, spectral_kurtosis=True, **kw)
        assert e.value.code == -2, (bin_e, kw)
