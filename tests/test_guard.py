"""Guard-bit transform (RTLSDR_GPU_FLAG_GUARD_BITS) without a GPU: the oracle (tests/oracle_guard.c) against a float64
DFT and against the int16 fix_fft where nothing rounds, every guard kernel through the CPU emulator
(tests/emu/guard_entry.cpp) against the oracle exactly, and the guard dB rows and their CSV text."""
import ctypes
import math
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
GUARD_SO = os.path.join(EMU_DIR, "libguard_emu.so")
ORACLE_GUARD_SO = os.path.join(ROOT, "tests", "liboracle_guard.so")
F = 8
SUM, PEAK, SK = 0, 1, 2
_oracle_guard_lib = None


def oracle_guard_lib():
    """tests/oracle_guard.c, built with the oracle's flags (asserts on: the int32 bound is checked)"""
    global _oracle_guard_lib
    if _oracle_guard_lib is None:
        src = os.path.join(ROOT, "tests", "oracle_guard.c")
        deps = [src] + [os.path.join(ROOT, "oracle", f) for f in ("scan_oracle.c", "scan_oracle.h")]
        if not os.path.exists(ORACLE_GUARD_SO) or any(os.path.getmtime(d) > os.path.getmtime(ORACLE_GUARD_SO)
                                                      for d in deps):
            subprocess.run(["gcc", "-O3", "-fwrapv", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "oracle"),
                            "-o", ORACLE_GUARD_SO, src, "-lm"], check=True)
        L = ctypes.CDLL(ORACLE_GUARD_SO)
        L.oracle_fix_fft_guard.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        L.oracle_scan_read_guard.argtypes = [ctypes.c_void_p] * 7
        L.oracle_guard_front_blocks.argtypes = [ctypes.c_void_p] * 4
        L.oracle_epilogue_guard.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_int,
                                            ctypes.c_int, ctypes.c_void_p]
        _oracle_guard_lib = L
    return _oracle_guard_lib


def _cfg(port_oracle, plan, window):
    sine = np.ascontiguousarray(np.concatenate([port_oracle.sine_table(plan["bin_e"]), np.zeros(4, np.int16)]))
    window = np.ascontiguousarray(window, dtype=np.int32)
    cfg = OracleCfg(plan["bin_e"], plan["buf_len"], plan["downsample"], plan["downsample_passes"], plan["boxcar"],
                    plan["comp_fir_size"], plan.get("peak_hold", 0), window.ctypes.data, sine.ctypes.data)
    return cfg, (sine, window)


def oracle_guard(port_oracle, plan, window, reads, hops, tune_count=None):
    """(avg [tc, N], samples [tc], s2 uint64 [tc, N, 2]) of the guard scan of `reads` (S2 only without peak hold)"""
    lib = oracle_guard_lib()
    n = 1 << plan["bin_e"]
    tc = tune_count or plan["tune_count"]
    cfg, keep = _cfg(port_oracle, plan, window)
    avg = np.zeros((tc, n), dtype=np.int64)
    samples = np.zeros(tc, dtype=np.int32)
    s2 = np.zeros((tc, n, 2), dtype=np.uint64)
    work = np.zeros(plan["buf_len"] + 16, dtype=np.int16)
    v = np.zeros(2 * n, dtype=np.int32)
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    for i, h in enumerate(hops):
        s = ctypes.c_int(int(samples[h]))
        lib.oracle_scan_read_guard(ctypes.addressof(cfg), _ptr(reads[i]), _ptr(work), _ptr(v), _ptr(avg[h]),
                                   ctypes.addressof(s), None if plan.get("peak_hold", 0) else _ptr(s2[h]))
        samples[h] = s.value
    return avg, samples, s2


def guard_db(avg, bin_e, crop, rate, samples):
    """the guard dB row of one hop (oracle_epilogue_guard)"""
    a = np.ascontiguousarray(avg, dtype=np.int64).copy()
    db = np.zeros((1 << bin_e) + 2, dtype=np.float64)
    k = oracle_guard_lib().oracle_epilogue_guard(_ptr(a), bin_e, crop, rate, int(samples), _ptr(db))
    return db[:k]


def guard_fft(port_oracle, x16, m):
    """oracle_fix_fft_guard of int16 (re, im) pairs x16 [2N]: int32 [2N]"""
    v = np.ascontiguousarray(x16.astype(np.int32) << F)
    sine = np.ascontiguousarray(np.concatenate([port_oracle.sine_table(m), np.zeros(4, np.int16)]))
    assert oracle_guard_lib().oracle_fix_fft_guard(_ptr(v), m, _ptr(sine), m) == 0
    return v


@pytest.fixture(scope="module")
def guard_emu():
    srcs = [os.path.join(EMU_DIR, f) for f in ("guard_entry.cpp", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".inl"))]
    srcs.append(os.path.join(ROOT, "include", "rtlsdr_gpu_scan.h"))
    if not os.path.exists(GUARD_SO) or any(os.path.getmtime(s) > os.path.getmtime(GUARD_SO) for s in srcs):
        subprocess.run(["g++", "-std=c++20", "-O2", "-ffp-contract=off", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC,
                        "-shared", "-fPIC", "-pthread", "-o", GUARD_SO, os.path.join(EMU_DIR, "guard_entry.cpp")],
                       check=True)
    return ctypes.CDLL(GUARD_SO)


# ---- the oracle ------------------------------------------------------------------------------------------

def dft_bound(m, amax):
    """Worst-case |guard - exact| per output (complex magnitude, in output units) after m stages.  A stage computes
    q + t with q = a >> 1 (floor: < 1/2 per component) and t from two products, each rounded (<= 1/2), so it adds
    < 1.5 per component, < 1.5 sqrt(2) < 2.2 in magnitude.  The halved Q15 twiddle differs from exp(-i theta) / 2 by
    < 1.75 / 2^15 per component (sine rounded to integers on a 32767 scale, then halved with a floor), < 2^-13.5 in
    magnitude, which adds < amax 2^-13.5 per stage.  A stage maps errors (ea, eb) to (ea + w eb) / 2 with |w| <= 1,
    so earlier errors do not grow, and no value exceeds amax = the largest input magnitude."""
    return m * (2.2 + amax * 2.0 ** -13.5) + 1e-9


def float64_fix_fft(port_oracle, z, m):
    """fix_fft's butterflies in float64 without rounding: the same permutation, the same halved Q15 twiddles (as
    exact doubles w / 2^15, doubled because R() divides by 2^15 and the stage halves) and the same halving"""
    n = 1 << m
    sine = port_oracle.sine_table(m).astype(np.int64)
    idx = np.arange(n)
    rev = np.zeros(n, dtype=np.int64)
    for b in range(m):
        rev |= ((idx >> b) & 1) << (m - 1 - b)
    x = z[rev].astype(np.complex128)
    for s in range(m):
        half = 1 << s
        g = np.arange(half)
        j = g << (m - 1 - s)
        wr = np.asarray(sine[j + n // 4] >> 1, dtype=np.float64)
        wi = np.asarray(np.asarray(-sine[j], dtype=np.int16) >> 1, dtype=np.float64)
        w = (wr + 1j * wi) / 2.0 ** 15
        x = x.reshape(-1, 2, half)
        a, b = x[:, 0, :], x[:, 1, :] * w
        x = np.stack([a / 2 + b, a / 2 - b], axis=1).reshape(-1)
    return x


def inputs(m):
    n = 1 << m
    rng = np.random.default_rng(m)
    full = np.full(2 * n, -32768)       # full scale on both components, and a full-scale alternating tone
    tone = np.tile([32767, 32767, -32768, -32768], n // 2 + 1)[:2 * n]
    return [rng.integers(-40, 41, 2 * n), rng.integers(-32768, 32768, 2 * n), full, tone]


@pytest.mark.parametrize("m", [1, 2, 3, 5, 8, 10, 12, 13, 14, 16, 17, 20, 21])
def test_oracle_guard_fft_rounding_bound(port_oracle, m):
    """against the same butterflies in float64: only the rounding differs, < 2.2 units per stage"""
    for x in inputs(m):
        x16 = x.astype(np.int16)
        got = guard_fft(port_oracle, x16, m)
        z = (x16[0::2].astype(np.float64) + 1j * x16[1::2].astype(np.float64)) * 2.0 ** F
        err = np.abs((got[0::2] + 1j * got[1::2]) - float64_fix_fft(port_oracle, z, m))
        assert err.max() <= m * 2.2, (m, err.max())


@pytest.mark.parametrize("m", [2, 3, 5, 8, 10, 12, 13, 14, 16, 17, 20, 21])
def test_oracle_guard_fft_matches_float64_dft(port_oracle, m):
    """against numpy's float64 DFT scaled by 2^F / N.  (N = 2 is not a DFT in fix_fft: its one twiddle is
    Sinewave[N/4] >> 1 = Sinewave[0] >> 1 = 0, so both outputs are a / 2; the bound test above covers it.)"""
    n = 1 << m
    for x in inputs(m):
        x16 = x.astype(np.int16)
        got = guard_fft(port_oracle, x16, m)
        z = x16[0::2].astype(np.float64) + 1j * x16[1::2].astype(np.float64)
        want = np.fft.fft(z) * (2.0 ** F / n)
        err = np.abs((got[0::2] + 1j * got[1::2]) - want)
        amax = np.abs(z).max() * 2.0 ** F
        assert err.max() <= dft_bound(m, amax), (m, err.max(), dft_bound(m, amax))


def test_oracle_guard_rounding_is_below_the_q15_paths(port_oracle):
    """low-level noise at 4096 bins: the guard transform's error against the DFT is far below the Q15 path's"""
    m, n = 12, 4096
    rng = np.random.default_rng(3)
    x16 = (rng.normal(0, 3, 2 * n) * 100).astype(np.int16)
    z = x16[0::2].astype(np.float64) + 1j * x16[1::2].astype(np.float64)
    exact = np.fft.fft(z) / n
    g = guard_fft(port_oracle, x16, m)
    q = port_oracle.fix_fft(x16.copy(), m)
    eg = np.abs((g[0::2] + 1j * g[1::2]) / 2.0 ** F - exact)
    eq = np.abs((q[0::2] + 1j * q[1::2]).astype(np.complex128) - exact)
    assert np.sqrt(np.mean(eg ** 2)) * 16 < np.sqrt(np.mean(eq ** 2))


def test_oracle_guard_equals_fix_fft_without_rounding(port_oracle):
    """N = 2: fix_fft's only twiddle is Sinewave[0] >> 1 = 0, so both outputs are a >> 1: nothing rounds, and the
    guard output >> F equals oracle_fix_fft exactly"""
    rng = np.random.default_rng(1)
    for _ in range(200):
        x16 = rng.integers(-32768, 32768, 4).astype(np.int16)
        g = guard_fft(port_oracle, x16, 1)
        q = port_oracle.fix_fft(x16.copy(), 1)
        assert np.array_equal(g >> F, q.astype(np.int32))


def test_oracle_guard_scan_is_the_sum_of_block_powers(port_oracle):
    bin_e, n = 6, 64
    plan = plan_dict(bin_e, tune_count=1)
    win = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=4, param=30)
    avg, smp, s2 = oracle_guard(port_oracle, plan, win, reads, hops)
    cfg, keep = _cfg(port_oracle, plan, win)
    tot, tot2 = [0] * n, [0] * n
    for r in reads:
        out = np.zeros(plan["buf_len"], dtype=np.int16)
        work = np.zeros(plan["buf_len"] + 16, dtype=np.int16)
        b = oracle_guard_lib().oracle_guard_front_blocks(ctypes.addressof(cfg), _ptr(r), _ptr(work), _ptr(out))
        for k in range(b):
            v = guard_fft(port_oracle, out[k * 2 * n:(k + 1) * 2 * n], bin_e)
            for j in range(n):
                pw = (int(v[2 * j]) ** 2 + int(v[2 * j + 1]) ** 2 + 128) >> F
                tot[j] += pw
                tot2[j] += pw * pw
    assert avg[0].tolist() == tot
    assert [int(lo) | (int(hi) << 64) for lo, hi in s2[0]] == tot2
    assert smp[0] == len(reads) * (plan["buf_len"] // (2 * n))


# ---- the guard kernels through the emulator ---------------------------------------------------------------

def full_scale(buf_len):
    b = np.zeros(buf_len, dtype=np.uint8)
    b[0::4] = b[1::4] = 255
    return b


def run_u8(guard_emu, port_oracle, plan, win, reads, hops, mode, grid, b_groups=1):
    bin_e, n, tc = plan["bin_e"], 1 << plan["bin_e"], plan["tune_count"]
    sreads, shops, _ = sort_by_hop(reads, hops, tc)
    shops = np.ascontiguousarray(shops, dtype=np.int32)
    avg = np.zeros((tc, n), dtype=np.int64)
    smp = np.zeros(tc, dtype=np.int64)
    s2 = np.zeros((tc, n, 2), dtype=np.uint64)
    sine = port_oracle.sine_table(bin_e)
    win = np.ascontiguousarray(win, dtype=np.int32)
    assert guard_emu.emu_guard_u8(bin_e, vp(sreads), len(sreads), plan["buf_len"], vp(shops), grid, b_groups, mode,
                                  vp(sine), vp(win), vp(avg), vp(smp), vp(s2)) == 0
    return avg, smp, s2


@pytest.mark.parametrize("bin_e", list(range(1, 13)))
def test_guard_small_u8_kernel(guard_emu, port_oracle, bin_e):
    """every bin count of the u8 path, the sum, peak-hold and SK instances, random windows and full-scale reads"""
    n = 1 << bin_e
    rng = np.random.default_rng(bin_e)
    for mode in (SUM, PEAK, SK):
        plan = plan_dict(bin_e, peak_hold=1 if mode == PEAK else 0, tune_count=2)
        win = rng.integers(-70000, 70000, n).astype(np.int32) if bin_e % 2 else port_oracle.window_coefs("hamming", n)
        reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=10)
        reads[1::2] = full_scale(16384)
        want_avg, want_smp, want_s2 = oracle_guard(port_oracle, plan, win, reads, hops)
        if mode == SK and bin_e % 2 == 0:   # (a random window spreads the tone's power over many bins)
            assert want_s2[..., 1].any(), "the full-scale reads must reach S2's high word"
        for grid in ((1, 5) if bin_e in (1, 12) else (3,)):
            avg, smp, s2 = run_u8(guard_emu, port_oracle, plan, win, reads, hops, mode, grid)
            assert np.array_equal(avg, want_avg), (mode, grid)
            assert np.array_equal(smp, want_smp), (mode, grid)
            if mode == SK:
                assert np.array_equal(s2, want_s2), grid


@pytest.mark.parametrize("bin_e,b_groups", [(13, 1), (14, 2), (17, 2)])
def test_guard_large_u8_kernels(guard_emu, port_oracle, bin_e, b_groups):
    """N > 4096: both kernels, the three accumulations, a hop change inside a CTA's run of reads"""
    n = 1 << bin_e
    for mode in (SUM, PEAK, SK):
        plan = plan_dict(bin_e, buf_len=2 * n, peak_hold=1 if mode == PEAK else 0, tune_count=2)
        win = port_oracle.window_coefs("blackman", n)
        reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=bin_e + mode, param=35)
        reads[2] = full_scale(2 * n)
        want_avg, want_smp, want_s2 = oracle_guard(port_oracle, plan, win, reads, hops)
        avg, smp, s2 = run_u8(guard_emu, port_oracle, plan, win, reads, hops, mode, 3, b_groups)
        assert np.array_equal(avg, want_avg), mode
        assert np.array_equal(smp, want_smp), mode
        if mode == SK:
            assert want_s2[..., 1].any()
            assert np.array_equal(s2, want_s2)


def decimated(emu, port_oracle, plan, reads, win):
    """the library's decimators (emulated) -> c16 images and DC sums, as test_sk.py takes them"""
    bin_e, n = plan["bin_e"], 1 << plan["bin_e"]
    box = plan["boxcar"] and plan["downsample"] > 1
    l_len = plan["buf_len"] // plan["downsample"]
    blocks = (l_len + 2 * n - 1) // (2 * n)
    padded = blocks
    while (padded * n) % 4:
        padded += 1
    images = np.zeros((len(reads), padded * n), dtype=np.uint32)
    sums = np.zeros((len(reads), 2), dtype=np.int64)
    segs = np.array([(0, 0, len(reads), 0)], dtype=np.int32)
    scratch = np.zeros((1, n), dtype=np.int64)
    sine = port_oracle.sine_table(bin_e)
    emu.emu_small_decim(bin_e, 0, vp(reads), len(reads), plan["buf_len"], plan["downsample"],
                        plan["downsample_passes"], 0 if box else 1, None, vp(segs), 1, vp(sine), vp(win),
                        vp(scratch), vp(images), vp(sums))
    return images, sums


LARGE_DECIMATED = {
    # one 2^13-point block per read behind a boxcar (ds = 2), and behind a -F 0 chain of two passes (ds = 4; the
    # emulated decimators here run without the compensation FIR, the GPU tests cover -F 9 at this size)
    "box13": plan_dict(13, buf_len=32768, downsample=2),
    "fir14": plan_dict(14, buf_len=131072, downsample=4, downsample_passes=2, boxcar=0, comp_fir_size=0),
}


@pytest.mark.parametrize("freq,fir", [("100M:100.1M:100", -1), ("100M:100.3M:3k", 5), ("100M:100.2M:1k", 0),
                                      ("box13", None), ("fir14", None)])
def test_guard_in16_kernel(emu, guard_emu, port_oracle, freq, fir):
    """decimated images: a narrow boxcar scan (ds = 28), -F 5 and -F 0, sum / peak / SK; and the large path
    (N >= 8192: both guard kernels) behind a boxcar and a -F chain"""
    from rtlsdr_b200.planner import plan_scan
    base = dict(LARGE_DECIMATED[freq]) if freq in LARGE_DECIMATED else plan_scan(freq, 0.0, None if fir < 0 else
                                                                               fir).as_dict()
    bin_e, n = base["bin_e"], 1 << base["bin_e"]
    box = base["boxcar"] and base["downsample"] > 1
    win = np.ascontiguousarray(port_oracle.window_coefs("hamming", n), dtype=np.int32)
    for mode in (SUM, PEAK, SK):
        plan = dict(base, peak_hold=1 if mode == PEAK else 0, tune_count=1)
        reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_XORSHIFT, seed=5 + mode)
        reads[1] = full_scale(plan["buf_len"])
        want_avg, want_smp, want_s2 = oracle_guard(port_oracle, plan, win, reads, hops)
        images, sums = decimated(emu, port_oracle, plan, reads, win)
        for grid in (1, 4):
            avg = np.zeros((1, n), dtype=np.int64)
            smp = np.zeros(1, dtype=np.int64)
            s2 = np.zeros((1, n, 2), dtype=np.uint64)
            hop_of = np.zeros(len(reads), dtype=np.int32)
            sine = port_oracle.sine_table(bin_e)
            assert guard_emu.emu_guard_in16(bin_e, vp(images), vp(sums), len(reads), plan["buf_len"],
                                            plan["downsample"], plan["downsample_passes"], 1 if box else 0,
                                            vp(hop_of), grid, 1, mode, vp(sine), vp(win), vp(avg), vp(smp),
                                            vp(s2)) == 0
            assert np.array_equal(avg, want_avg), (mode, grid)
            assert np.array_equal(smp, want_smp), (mode, grid)
            if mode == SK:
                assert np.array_equal(s2, want_s2), grid


# ---- dB rows and their text -----------------------------------------------------------------------------------

def guard_report_cases(rng, bin_e):
    n = 1 << bin_e
    avg = rng.integers(0, 1 << 62, (4, n)).astype(np.int64)
    avg[1] = rng.integers(0, 3, n)                  # the smallest non-zero bins
    avg[2, :] = (1 << 63) - 1
    smp = np.array([40, (1 << 31) - 1, 1, 0], dtype=np.int64)
    return avg, smp


@pytest.mark.parametrize("bin_e,crop,rate", [(1, 0.0, 2400000), (10, 0.3, 2147483647), (12, 0.2, 1000)])
def test_guard_epilogue_matches_oracle(guard_emu, bin_e, crop, rate):
    rng = np.random.default_rng(bin_e)
    avg, smp = guard_report_cases(rng, bin_e)
    n = 1 << bin_e
    i1, i2 = int(n * crop * 0.5), (n - 1) - int(n * crop * 0.5)
    got = np.zeros((4, i2 - i1 + 2))
    guard_emu.emu_guard_epilogue(vp(avg), vp(smp), vp(got), bin_e, i1, i2, rate, 4)
    for h in range(4):
        want = guard_db(avg[h], bin_e, crop, rate, int(smp[h]))
        assert got[h].tobytes() == want.tobytes(), h


def test_guard_epilogue_iir(guard_emu):
    """-s iir on a guard handle: the smoothing runs on the scaled linear value d = avg * 2^-8 / rate / samples,
    s = d at a bin's first report, s += alpha (d - s) after it, a report without samples prints d and keeps s"""
    bin_e, rate, alpha = 6, 2400000, 0.25
    n, rng = 1 << bin_e, np.random.default_rng(4)
    count = n + 1
    state = np.full((1, n), np.nan)
    s = np.full(n, np.nan)
    for rep in range(4):
        avg = rng.integers(1, 1 << 40, (1, n)).astype(np.int64)
        smp = np.array([0 if rep == 2 else 7 * (rep + 1)], dtype=np.int64)
        got = np.zeros((1, count))
        guard_emu.emu_guard_epilogue_iir(vp(avg), vp(smp), vp(got), bin_e, 0, n - 1, rate, 1, vp(state),
                                         ctypes.c_double(alpha))
        want = []
        for i in range(n):
            j = (i + n // 2) & (n - 1)
            v = float(avg[0, 1 if j == 0 else j])
            d = v * 2.0 ** -8 / float(rate) / float(smp[0]) if smp[0] else math.inf  # (a bin > 0 over no samples)
            if smp[0]:
                s[i] = d if s[i] != s[i] else s[i] + alpha * (d - s[i])
                want.append(10 * math.log10(s[i]))
            else:
                want.append(10 * math.log10(d))
        want.append(want[-1])
        assert np.array_equal(got[0], np.array(want), equal_nan=True), rep


def test_guard_rows_stay_inside_the_csv_formatters_domain(guard_emu):
    """the lowest guard value (a bin of 1 after 2^31 - 1 samples at rate 2^31 - 1) is -210.7 dB and the highest
    below 190 dB: both within the 7 characters ("-999.99") the row kernels print"""
    avg = np.array([[1, 1], [(1 << 63) - 1, (1 << 63) - 1]], dtype=np.int64)
    smp = np.array([(1 << 31) - 1, 1], dtype=np.int64)
    got = np.zeros((2, 3))
    guard_emu.emu_guard_epilogue(vp(avg), vp(smp), vp(got), 1, 0, 1, 2147483647, 2)
    assert -211 < got[0].min() < -210 and got[1].max() < 190


def test_guard_csv_text_matches_printf(guard_emu, port_oracle):
    """guard dB rows -- including the lowest values the domain allows -- through the GPU row formatter equal
    host printf("%.2f") of the oracle's doubles"""
    import test_csv_text as tc
    from rtlsdr_b200.planner import plan_scan
    lib = csv_row_emu()
    plan = plan_scan("88M:108M:1k", 0.2, None)
    assert plan.tune_count >= 3
    rng = np.random.default_rng(9)
    rows = 3
    n = 1 << plan.bin_e
    avg = rng.integers(0, 1 << 40, (rows, n)).astype(np.int64)
    avg[1] = 1
    smp = np.array([1000, (1 << 31) - 1, 7], dtype=np.int32)
    db = np.stack([guard_db(avg[r], plan.bin_e, plan.crop, 2147483647, int(smp[r])) for r in range(rows)])
    assert db.shape[1] == plan.db_count and db.min() < -200
    n_out, text = tc.emu_rows(lib, plan, 0, rows, np.ascontiguousarray(db), smp)
    want = "".join(tc.STAMP + plan.csv_row(r, int(smp[r]), db[r]) for r in range(rows))
    assert text[:n_out].tobytes().decode() == want


def csv_row_emu():
    """tests/emu/csv_entry.cpp: the CSV row kernels through the emulator"""
    so = os.path.join(EMU_DIR, "libcsv_guard_emu.so")
    srcs = [os.path.join(EMU_DIR, "csv_entry.cpp")] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-std=c++20", "-O2", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC, "-shared", "-fPIC",
                        "-pthread", "-o", so, os.path.join(EMU_DIR, "csv_entry.cpp")], check=True)
    L = ctypes.CDLL(so)
    i64, p = ctypes.c_longlong, ctypes.c_void_p
    L.emu_csv_rows.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, p, i64, p, p, p, ctypes.c_int,
                               ctypes.c_double, ctypes.c_int, p]
    L.emu_csv_rows.restype = i64
    return L


def test_guard_config_errors_before_any_device_work():
    """guard bits on the rms path (bin_e 0): RTLSDR_GPU_ERR_CONFIG"""
    import rtlsdr_b200.scan as rs
    from rtlsdr_b200 import _build
    _build.build_cuda()
    with pytest.raises(rs.ScanError) as e:
        rs.GpuScan(2, 0, 16384, guard_bits=True)
    assert e.value.code == -2
