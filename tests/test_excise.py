"""Spectral-kurtosis RFI excision (RTLSDR_GPU_FLAG_SK_EXCISION) without a GPU: sk.cuh's sk_sigma() against its
closed form and a Monte Carlo variance, excise.cuh's fold and report kernels through the CPU emulator
(tests/emu/excise_entry.cpp) against a Python oracle bit for bit, the report rows' text against host printf, and
init's refusal of the flag without spectral kurtosis."""
import ctypes
import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")
U64 = (1 << 64) - 1
U128 = (1 << 128) - 1
STAMP = "2026-01-01, 00:00:00, "
ROW_FIXED, VALUE_MAX, F4_VALUE_MAX = 56, 9, 17
INF = float("inf")


def vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def ex(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("excise_emu") / "libexcise_emu.so")
    subprocess.run(["g++", "-std=c++20", "-O2", "-ffp-contract=off", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC,
                    "-shared", "-fPIC", "-pthread", "-o", so, os.path.join(EMU_DIR, "excise_entry.cpp")], check=True)
    L = ctypes.CDLL(so)
    p, i, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    L.emu_sk_sigma.argtypes = [ctypes.c_int64]
    L.emu_sk_sigma.restype = d
    L.emu_sk_from_moments.argtypes = [ctypes.c_int64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int64]
    L.emu_sk_from_moments.restype = d
    L.emu_excise_fold.argtypes = [p] * 9 + [d, d, i, i, i]
    L.emu_excise_fold.restype = None
    L.emu_excised_report.argtypes = [i] + [p] * 6 + [i] * 6
    L.emu_excised_report.restype = None
    L.emu_rows.argtypes = [i, ctypes.c_char_p, i, p, i, p, p, p, d, p]
    L.emu_rows.restype = ctypes.c_longlong
    return L


def same_bits(a, b):
    return np.float64(a).tobytes() == np.float64(b).tobytes()


# ---- sk_sigma ------------------------------------------------------------------------------------------

def test_sk_sigma_closed_form(ex):
    for M in list(range(-3, 300)) + [1000, 4095, 65536, 1 << 20, (1 << 31) - 1, 1 << 40]:
        got = ex.emu_sk_sigma(M)
        if M < 2:
            assert math.isnan(got), M
            continue
        m = float(M)
        want = math.sqrt((4.0 * m * m) / (((m - 1.0) * (m + 2.0)) * (m + 3.0)))
        assert same_bits(got, want), M                          # the header's fixed order in IEEE doubles
        exact = Fraction(4 * M * M, (M - 1) * (M + 2) * (M + 3))
        assert abs(Fraction(got) ** 2 - exact) <= exact * Fraction(1, 1 << 50), M


@pytest.mark.parametrize("M", [16, 64, 256])
def test_sk_sigma_against_monte_carlo(ex, M):
    """single-block power of Gaussian noise is exponential; the spread of SK over many sub-integrations is sigma"""
    rng = np.random.default_rng(M)
    trials = 40000
    pw = rng.exponential(1.0, (trials, M))
    s1, s2 = pw.sum(1), (pw * pw).sum(1)
    sk = (M + 1) / (M - 1) * (M * s2 / (s1 * s1) - 1)
    sigma = ex.emu_sk_sigma(M)
    # the standard error of a standard deviation from n samples is about sigma * sqrt(kurtosis / 4n)
    assert abs(sk.std() / sigma - 1) < 0.03, (sk.std(), sigma)
    assert abs(sk.mean() - 1) < 5 * sigma / math.sqrt(trials)


# ---- oracle --------------------------------------------------------------------------------------------

class State:
    """one handle's accumulators and excision state as Python integers"""

    def __init__(self, hops, n):
        self.hops, self.n = hops, n
        self.S1 = [[0] * n for _ in range(hops)]
        self.S2 = [[0] * n for _ in range(hops)]
        self.smp = [0] * hops
        self.snap1 = [[0] * n for _ in range(hops)]
        self.snap2 = [[0] * n for _ in range(hops)]
        self.c1 = [[0] * n for _ in range(hops)]
        self.b1 = [[0] * n for _ in range(hops)]
        self.snap_smp = [0] * hops

    def zero(self):
        self.__init__(self.hops, self.n)


def fold_oracle(ex, st, k_low, k_high, ds):
    for h in range(st.hops):
        M = (st.smp[h] - st.snap_smp[h]) // ds
        sig = ex.emu_sk_sigma(M)
        lo, hi = 1.0 - k_low * sig, 1.0 + k_high * sig       # NaN for M < 2: nothing flags
        for j in range(st.n):
            d1 = st.S1[h][j] - st.snap1[h][j]
            d2 = (st.S2[h][j] - st.snap2[h][j]) & U128
            sk = ex.emu_sk_from_moments(d1, d2 & U64, d2 >> 64, M)
            if not (sk == sk and (sk < lo or sk > hi)):
                st.c1[h][j] += d1
                st.b1[h][j] += M
            st.snap1[h][j], st.snap2[h][j] = st.S1[h][j], st.S2[h][j]
        st.snap_smp[h] = st.smp[h]


def report_oracle(st, bin_e, i1, i2, rate, ds, guard):
    n, count = 1 << bin_e, i2 - i1 + 2
    db = np.zeros((st.hops, count))
    fl = np.zeros((st.hops, count))
    for h in range(st.hops):
        F = st.snap_smp[h] // ds
        for k in range(count):
            i = i1 + k if k < count - 1 else i2
            j = (i + n // 2) & (n - 1)
            j = 1 if j == 0 else j
            v, B = st.c1[h][j], st.b1[h][j]
            if B == 0:
                d = float("nan")
            else:
                x = float(v) * 2.0 ** -8 if guard else float(v)
                s = float(B * ds)
                d = x / float(rate) / s if k < count - 1 else x / (float(rate) * s)
                d = 10 * math.log10(d) if d > 0 else -INF
            db[h, k] = d
            fl[h, k] = float("nan") if F == 0 else float(F - B) / float(F)
    return db, fl


def to_arrays(st):
    tc, n = st.hops, st.n
    a = lambda rows, dt: np.array(rows, dtype=dt).reshape(tc, -1)  # noqa: E731
    s2 = np.zeros((tc, n, 2), np.uint64)
    ss2 = np.zeros((tc, n, 2), np.uint64)
    for h in range(tc):
        for j in range(n):
            s2[h, j] = (st.S2[h][j] & U64, st.S2[h][j] >> 64)
            ss2[h, j] = (st.snap2[h][j] & U64, st.snap2[h][j] >> 64)
    return dict(avg=a(st.S1, np.int64), s2=s2, smp=np.array(st.smp, np.int64), snap1=a(st.snap1, np.int64),
                snap2=ss2, c1=a(st.c1, np.int64), b1=a(st.b1, np.int32), snap_smp=np.array(st.snap_smp, np.int64))


def emu_fold(ex, dev, bin_e, ds, k_low, k_high):
    ticket = np.zeros(dev["smp"].size, np.uint32)
    ex.emu_excise_fold(vp(dev["avg"]), vp(dev["smp"]), vp(dev["s2"]), vp(dev["snap1"]), vp(dev["snap2"]),
                       vp(dev["c1"]), vp(dev["b1"]), vp(dev["snap_smp"]), vp(ticket), k_low, k_high, bin_e, ds,
                       dev["smp"].size)
    assert not ticket.any()


def emu_report(ex, dev, bin_e, i1, i2, rate, ds, guard):
    tc, count = dev["smp"].size, i2 - i1 + 2
    smp = np.zeros(tc, np.int32)
    db = np.zeros((tc, count))
    fl = np.zeros((tc, count))
    ex.emu_excised_report(int(guard), vp(dev["c1"]), vp(dev["b1"]), vp(dev["snap_smp"]), vp(smp), vp(db), vp(fl),
                          bin_e, i1, i2, rate, ds, tc)
    return smp, db, fl


def add_sub_integration(st, rng, M, ds, kind):
    """M more FFT blocks into every bin of every hop: noise, bursts, steady tones, empty bins"""
    for h in range(st.hops):
        m = M[h]
        pw = rng.exponential(1 << 18, (st.n, m)).astype(np.int64)
        if kind == "burst":
            pw[:: 3, : max(1, m // 8)] *= 40                  # SK > 1 in every third bin
        elif kind == "steady":
            pw[1:: 3] = (1 << 20) + rng.integers(0, 64, (pw[1:: 3].shape))   # SK < 1
        pw[2:: 7] = 0                                         # dS1 = 0
        d1 = pw.sum(1)
        d2 = (pw * pw).sum(1)
        for j in range(st.n):
            st.S1[h][j] += int(d1[j])
            st.S2[h][j] += int(d2[j])
        st.smp[h] += m * ds


def check_against_oracle(ex, st, bin_e, i1, i2, rate, ds, guard, k_low, k_high):
    dev = to_arrays(st)
    emu_fold(ex, dev, bin_e, ds, k_low, k_high)
    fold_oracle(ex, st, k_low, k_high, ds)
    want = to_arrays(st)
    for key in ("snap1", "snap2", "c1", "b1", "snap_smp"):
        assert np.array_equal(dev[key], want[key]), key
    smp, db, fl = emu_report(ex, dev, bin_e, i1, i2, rate, ds, guard)
    assert np.array_equal(smp, want["snap_smp"].astype(np.int32))
    wdb, wfl = report_oracle(st, bin_e, i1, i2, rate, ds, guard)
    assert db.tobytes() == wdb.tobytes()
    assert fl.tobytes() == wfl.tobytes()
    return db, fl


@pytest.mark.parametrize("bin_e,hops,ds,guard,i1,i2", [
    (3, 2, 1, False, 0, 7),        # every bin, DC nuke at i = n/2, duplicate of the last
    (5, 3, 3, True, 4, 27),        # crop, decimated counts, guard-bit scaling
    (9, 2, 2, False, 100, 411),    # two CTAs per hop
])
def test_fold_and_report_match_oracle(ex, bin_e, hops, ds, guard, i1, i2):
    rng = np.random.default_rng(bin_e * 31 + hops)
    n = 1 << bin_e
    st = State(hops, n)
    # S2 just below a multiple of 2^64 at the last fold: the next difference borrows out of the low word
    for h in range(hops):
        for j in range(n):
            base2 = ((h + 1) << 64) + U64 - int(rng.integers(0, 1 << 20))
            base1 = int(rng.integers(0, 1 << 40))
            st.S1[h][j] = st.snap1[h][j] = base1
            st.S2[h][j] = st.snap2[h][j] = base2
    rate = 2400000
    plan = [  # (M per hop, kind, k_low, k_high)
        ([64] * hops, "burst", 3.0, 3.0),
        ([1] + [2] * (hops - 1), "noise", 3.0, 3.0),           # M < 2 never flags; M = 2 at its edge
        ([0] + [128] * (hops - 1), "steady", 3.0, 3.0),        # a hop without reads since the last fold
        ([96] * hops, "steady", INF, 2.0),                     # k_low = +inf keeps steady carriers
        ([80] * hops, "burst", 0.0, INF),                      # k_high = +inf keeps bursts
    ]
    flagged_any = False
    for M, kind, kl, kh in plan:
        add_sub_integration(st, rng, M, ds, kind)
        db, fl = check_against_oracle(ex, st, bin_e, i1, i2, rate, ds, guard, kl, kh)
        flagged_any |= bool(np.nanmax(fl) > 0)
    assert flagged_any
    # a read-and-zero clears the state with the sums; folding goes on from zero
    st.zero()
    add_sub_integration(st, rng, [64] * hops, ds, "burst")
    check_against_oracle(ex, st, bin_e, i1, i2, rate, ds, guard, 3.0, 3.0)


def test_report_of_a_fresh_state_is_nan(ex):
    st = State(2, 8)
    dev = to_arrays(st)
    smp, db, fl = emu_report(ex, dev, 3, 0, 7, 2400000, 1, False)
    assert not smp.any()
    assert np.isnan(db).all() and not np.signbit(db).any()
    assert np.isnan(fl).all()


# ---- text ----------------------------------------------------------------------------------------------

def host_row(stamp, low, high, step, smp, vals, f4):
    head = "%s%i, %i, %.2f, %i, " % (stamp, low, high, step, smp)
    fmt = "%.4f" if f4 else "%.2f"
    return head + ", ".join("nan" if math.isnan(v) else fmt % v for v in vals) + "\n"


@pytest.mark.parametrize("guard", [False, True])
def test_excised_rows_text_matches_printf(ex, guard):
    rng = np.random.default_rng(5)
    bin_e, hops, ds = 5, 3, 2
    st = State(hops, 1 << bin_e)
    add_sub_integration(st, rng, [64, 0, 100], ds, "burst")
    fold_oracle(ex, st, 2.0, 2.0, ds)
    add_sub_integration(st, rng, [64, 0, 100], ds, "steady")   # hop 1 never read: NaN rows
    fold_oracle(ex, st, 2.0, 2.0, ds)
    st.c1[0][5] = 0                                           # -inf
    st.c1[2][7], st.b1[2][7] = (1 << 62), 1                   # the loudest bin
    dev = to_arrays(st)
    smp, db, fl = emu_report(ex, dev, bin_e, 2, 29, 2400000, ds, guard)
    assert np.isnan(db).any() and np.isinf(db).any()
    low = np.array([88000000, 89000000, 90000000], np.int32)
    high = low + 1000000
    step = 31250.0
    for f4, vals, width in ((0, db, VALUE_MAX), (1, fl, F4_VALUE_MAX)):
        cap = hops * (len(STAMP) + ROW_FIXED + width * vals.shape[1])
        text = np.zeros(cap, np.uint8)
        n = ex.emu_rows(f4, STAMP.encode(), hops, vp(np.ascontiguousarray(vals)), vals.shape[1], vp(smp), vp(low),
                        vp(high), step, vp(text))
        want = "".join(host_row(STAMP, low[r], high[r], step, smp[r], vals[r], f4) for r in range(hops))
        assert n == len(want)
        assert text[:n].tobytes().decode() == want


# ---- the library without a GPU -------------------------------------------------------------------------

def test_init_rejects_excision_without_sk_before_device_work():
    from rtlsdr_b200 import _build
    import rtlsdr_b200.scan as rs
    _build.build_cuda()
    lib = rs.load_library()

    def init(flags, **kw):
        cfg = rs._Cfg()
        cfg.struct_size = ctypes.sizeof(rs._Cfg)
        base = dict(device=0, tune_count=1, bin_e=10, buf_len=16384, downsample=1, downsample_passes=0,
                    boxcar=1, comp_fir_size=0, peak_hold=0, rate=2400000, crop=0.0, flags=flags)
        base.update(kw)
        for k, v in base.items():
            setattr(cfg, k, v)
        h = ctypes.c_void_p()
        rc = lib.rtlsdr_gpu_scan_init(ctypes.byref(cfg), ctypes.byref(h))
        if rc == 0:
            lib.rtlsdr_gpu_scan_close(h)
        return rc

    assert init(32) == -2                        # RTLSDR_GPU_ERR_CONFIG: excision needs spectral kurtosis
    assert init(32 | 16) == -2
    assert init(32 | 8, peak_hold=1) == -2       # every SK restriction applies
    assert init(32 | 8 | 2) == -2                # no ASYNC_REPORT
    assert init(32 | 8, bin_e=0, buf_len=16384) == -2
    import torch
    if not torch.cuda.is_available():
        assert init(32 | 8) in (-5, -6)          # a valid configuration reaches the device check
    assert lib.rtlsdr_gpu_scan_excise_fold(None, 3.0, 3.0) == -1
    assert lib.rtlsdr_gpu_scan_excised_report(None, None, None, None, None, None) == -1
