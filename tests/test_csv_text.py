"""rtl_power's CSV rows formatted on the GPU (rtlsdr_b200/csrc/csv_text.cuh) against the host's printf.

CPU: the device formatter compiled with g++ against tests/emu/cuda_emu.h, compared with glibc's snprintf on
>= 10 M values of every class a report can hold and beyond, and both row kernels run under the emulator against
stamp + rp_csv_row.  GPU: collect_csv / format_csv_device against collect_all + Plan.csv_row on twin handles fed
the same reads."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")
STAMP = "2026-01-01, 00:00:00, "
ROW_FIXED, VALUE_MAX = 56, 9


def vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def csv_emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("csv_emu") / "libcsv_emu.so")
    subprocess.run(["g++", "-std=c++20", "-O2", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC, "-shared", "-fPIC",
                    "-pthread", "-o", so, os.path.join(EMU_DIR, "csv_entry.cpp")], check=True)
    L = ctypes.CDLL(so)
    i64, p = ctypes.c_longlong, ctypes.c_void_p
    L.emu_csv_check_f2.argtypes = [p, i64, ctypes.POINTER(i64)]
    L.emu_csv_check_f2.restype = i64
    L.emu_csv_check_i.argtypes = [p, i64, ctypes.POINTER(i64)]
    L.emu_csv_check_i.restype = i64
    L.emu_csv_f2.argtypes = [ctypes.c_double, ctypes.c_char_p]
    L.emu_csv_rows.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, p, i64, p, p, p, ctypes.c_int,
                               ctypes.c_double, ctypes.c_int, p]
    L.emu_csv_rows.restype = i64
    return L


def value_classes(rng, n_uniform=6_000_000, n_bits=3_000_000):
    """every class of double the formatter is specified for"""
    parts = [rng.uniform(-200, 200, n_uniform)]
    # random bit patterns below 2^53: any sign, mantissa, and biased exponent up to 1075
    bits = rng.integers(0, 1 << 52, n_bits, dtype=np.uint64)
    bits |= rng.integers(0, 1076, n_bits, dtype=np.uint64) << np.uint64(52)
    bits |= rng.integers(0, 2, n_bits, dtype=np.uint64) << np.uint64(63)
    parts.append(bits.view(np.float64))
    parts.append(np.arange(-1600, 1601) / 8.0)                    # every exact tie k/8 in +-200
    bound = (np.arange(-20000, 20000) + 0.5) / 100.0              # rounding boundaries (k + 1/2)/100
    parts += [bound, np.nextafter(bound, np.inf), np.nextafter(bound, -np.inf)]
    parts.append(-rng.uniform(0, 0.01, 500_000))                  # small negative values
    sub = rng.integers(1, 1 << 52, 500_000, dtype=np.uint64)      # subnormals of both signs
    sub[::2] |= np.uint64(1) << np.uint64(63)
    parts.append(sub.view(np.float64))
    top = np.float64(2.0 ** 53)
    parts.append(np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, np.nextafter(top, 0), -np.nextafter(top, 0),
                           5e-324, -5e-324, 0.005, -0.005, 0.015, 0.025, 1e-3, 2.0 ** -10, 2.0 ** -11]))
    nan_bits = np.array([0x7FF0000000000001, 0x7FF8000000000000, 0xFFF8000000000000, 0xFFFFFFFFFFFFFFFF],
                        dtype=np.uint64)
    parts.append(nan_bits.view(np.float64))
    return np.ascontiguousarray(np.concatenate(parts))


def test_f2_matches_printf(csv_emu):
    v = value_classes(np.random.default_rng(1))
    assert v.size >= 10_000_000
    first = ctypes.c_longlong()
    bad = csv_emu.emu_csv_check_f2(vp(v), v.size, ctypes.byref(first))
    assert bad == 0, f"{bad} mismatches, first {v[first.value]!r}"


def test_f2_domain_edge(csv_emu):
    buf = ctypes.create_string_buffer(32)
    for x in (2.0 ** 53, -2.0 ** 53, 1e300, -1.7e308):
        assert csv_emu.emu_csv_f2(x, buf) == -1
    assert csv_emu.emu_csv_f2(-0.0, buf) == 5 and buf.value == b"-0.00"
    assert csv_emu.emu_csv_f2(-np.nan, buf) == 4 and buf.value == b"-nan"


def test_int_matches_printf(csv_emu):
    v = np.concatenate([np.array([-2 ** 31, 2 ** 31 - 1, 0, -1, 1, 9, 10, -10], dtype=np.int32),
                        np.random.default_rng(2).integers(-2 ** 31, 2 ** 31, 100_000).astype(np.int32)])
    first = ctypes.c_longlong()
    assert csv_emu.emu_csv_check_i(vp(v), v.size, ctypes.byref(first)) == 0, v[first.value]


def report_values(rng, rows, db_count):
    """dB rows as a report holds them: finite values in (-187, 190), -inf bins, and NaN rows (no samples)"""
    db = rng.uniform(-187, 190, (rows, db_count))
    db[:, rng.integers(0, db_count, max(1, db_count // 50))] = -np.inf
    smp = rng.integers(0, 1 << 20, rows).astype(np.int32)
    if rows > 1:
        db[1] = np.float64(np.nan)
        smp[1] = 0
    return np.ascontiguousarray(db), smp


def emu_rows(csv_emu, plan, row_first, rows, db, smp, stamp=STAMP):
    low, high, step = plan.csv_columns()
    cap = rows * (len(stamp) + ROW_FIXED + VALUE_MAX * db.shape[1])
    text = np.zeros(cap, dtype=np.uint8)
    n = csv_emu.emu_csv_rows(stamp.encode(), row_first, rows, vp(db), db.shape[1], vp(smp), vp(low), vp(high),
                             low.size, step, db.shape[1], vp(text))
    return n, text


@pytest.mark.parametrize("rng_,crop,fir", [("88M:108M:1M", 0.0, None), ("88M:108M:1M", 0.2, None),
                                           ("100M:102M:2.5k", 0.0, None), ("100M:102M:2.5k", 0.2, None),
                                           ("88M:108M:1k", 0.0, None), ("88M:108M:1k", 0.2, None),
                                           ("100M:101M:10", 0.0, None), ("100M:101M:10", 0.2, None),
                                           ("100M:100.2M:10", 0.0, 9), ("100M:100.3M:300", 0.2, 9)])
def test_row_kernels_match_rp_csv_row(csv_emu, rng_, crop, fir):
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(rng_, crop, fir)
    rng = np.random.default_rng(plan.bin_e)
    row_first = 1 if plan.tune_count > 3 else 0
    rows = min(plan.tune_count - row_first, 3)
    db, smp = report_values(rng, rows, plan.db_count)
    n, text = emu_rows(csv_emu, plan, row_first, rows, db, smp)
    want = "".join(STAMP + plan.csv_row(row_first + r, int(smp[r]), db[r]) for r in range(rows))
    assert n == len(want)
    assert text[:n].tobytes().decode() == want


def test_capacity_bound_is_tight_for_the_widest_row(csv_emu):
    """the longest row the domain allows: INT32_MIN edges and counts, the widest step, every value 7 wide"""
    db = np.full((1, 2), -999.99)
    smp = np.array([-2 ** 31], dtype=np.int32)
    low = high = smp
    cap = len(STAMP) + ROW_FIXED + VALUE_MAX * 2
    text = np.zeros(cap, dtype=np.uint8)
    step = np.nextafter(2.0 ** 31, 0)
    n = csv_emu.emu_csv_rows(STAMP.encode(), 0, 1, vp(db), 2, vp(smp), vp(low), vp(high), low.size, step, 2,
                             vp(text))
    want = "%s%i, %i, %.2f, %i, -999.99, -999.99\n" % (STAMP, low[0], high[0], step, smp[0])
    assert len(want) <= cap and cap - len(want) <= 3
    assert n == len(want) and text[:n].tobytes().decode() == want
    # one value wider than 7 characters, or outside |v| < 2^53, is an error, never text
    for bad in (-1000.0, 10000.0, 1e300):
        db[0, 1] = bad
        assert csv_emu.emu_csv_rows(STAMP.encode(), 0, 1, vp(db), 2, vp(smp), vp(low), vp(high), low.size, step,
                                    2, vp(text)) == -1


# ---- GPU ---------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def scan_mod():
    import rtlsdr_b200.scan as s
    s.load_library()
    return s


def twins(scan_mod, port_oracle, freq_range, crop=0.0, fir=None, peak=0, window="hamming", hops=None, **kw):
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(freq_range, crop, fir)
    pd = plan.as_dict()
    pd["peak_hold"] = peak
    w = port_oracle.window_coefs(window, 1 << pd["bin_e"]) if pd["bin_e"] else None
    a = scan_mod.GpuScan.from_plan(pd, window_coefs=w, hops=hops, **kw)
    b = scan_mod.GpuScan.from_plan(pd, window_coefs=w, hops=hops, **kw)
    b.set_csv_columns(*plan.csv_columns(hops))
    return plan, pd, a, b


def feed(port_oracle, pd, handles, sweeps, mode, seed, hop_first=0, hop_count=None, const=None):
    import torch
    from oracles import SYNTH_XORSHIFT
    from scan_cases import make_reads
    tc, b = pd["tune_count"], pd["buf_len"]
    reads, _ = make_reads(port_oracle.lib, pd, sweeps, mode if mode is not None else SYNTH_XORSHIFT, seed)
    if const is not None:
        reads[:] = const
    dev = torch.from_numpy(np.ascontiguousarray(reads)).cuda()
    hop_count = handles[0].tune_count if hop_count is None else hop_count
    for g in handles:
        g.submit_device(hop_first, hop_count, sweeps, dev.data_ptr() + hop_first * b, tc * b, b)
        g.sync()


def want_text(plan, a, hop0=0):
    _, smp, db = a.collect_all()
    return "".join(STAMP + plan.csv_row(hop0 + h, int(smp[h]), db[h]) for h in range(a.tune_count)).encode()


CONFIGS = [("100M:102.4M:2400", 0.0, None, "rectangle", 4), ("88M:108M:1k", 0.2, None, "hamming", 3),
           ("24M:1766M:1k", 0.0, 9, "hamming", 1), ("100M:102.4M:19", 0.0, None, "blackman-harris", 2),
           ("24M:1457.6M:700", 0.0, None, "hamming", 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", range(1, 6))
def test_collect_csv_configs(scan_mod, port_oracle, cfg):
    from oracles import SYNTH_BIASED
    rng_, crop, fir, window, sweeps = CONFIGS[cfg - 1]
    plan, pd, a, b = twins(scan_mod, port_oracle, rng_, crop, fir, peak=1 if cfg == 4 else 0, window=window)
    feed(port_oracle, pd, (a, b), sweeps, SYNTH_BIASED, cfg)
    assert b.collect_csv(STAMP) == want_text(plan, a)
    assert b.collect_csv(STAMP) == want_text(plan, a)   # read-and-zero: the next report is empty (nan rows)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["peak", "rms", "const127", "hop_without_reads", "partial_hops"])
def test_collect_csv_cases(scan_mod, port_oracle, case):
    from oracles import SYNTH_XORSHIFT
    hops = range(2, 7) if case == "partial_hops" else None
    rng_ = "88M:108M:1M" if case == "rms" else "88M:108M:2.5k"
    plan, pd, a, b = twins(scan_mod, port_oracle, rng_, 0.2, peak=int(case == "peak"), hops=hops)
    if case == "partial_hops":
        # a -t worker's shard: the handle's hop i is the plan's hop 2 + i
        import torch
        from scan_cases import make_reads
        reads, _ = make_reads(port_oracle.lib, pd, 2, SYNTH_XORSHIFT, 5)
        dev = torch.from_numpy(reads).cuda()
        for g in (a, b):
            g.submit_device(0, len(hops), 2, dev.data_ptr() + hops.start * pd["buf_len"],
                            pd["tune_count"] * pd["buf_len"], pd["buf_len"])
            g.sync()
        assert b.collect_csv(STAMP) == want_text(plan, a, hops.start)
        return
    feed(port_oracle, pd, (a, b), 2, SYNTH_XORSHIFT, 4, hop_first=1 if case == "hop_without_reads" else 0,
         hop_count=pd["tune_count"] - 1 if case == "hop_without_reads" else None,
         const=127 if case == "const127" else None)
    text = b.collect_csv(STAMP)
    assert text == want_text(plan, a)
    if case == "const127":
        assert b"-inf" in text


@pytest.mark.gpu
def test_collect_csv_iir_three_reports(scan_mod, port_oracle):
    from oracles import SYNTH_BIASED
    plan, pd, a, b = twins(scan_mod, port_oracle, "88M:108M:1k", 0.2, iir_alpha=0.25)
    for rep in range(3):
        feed(port_oracle, pd, (a, b), 2, SYNTH_BIASED, 10 + rep)
        assert b.collect_csv(STAMP) == want_text(plan, a), rep


@pytest.mark.gpu
def test_format_csv_device_and_errors(scan_mod, port_oracle):
    import torch
    from oracles import SYNTH_BIASED
    from rtlsdr_b200.scan import ScanError
    plan, pd, a, b = twins(scan_mod, port_oracle, "88M:108M:1k", 0.2)
    c = scan_mod.GpuScan.from_plan(pd, window_coefs=port_oracle.window_coefs("hamming", 4096))
    c.set_csv_columns(*plan.csv_columns())
    feed(port_oracle, pd, (a, b, c), 2, SYNTH_BIASED, 7)
    tc, dc = pd["tune_count"], c.db_count
    db = torch.zeros(tc, dc, dtype=torch.float64, device="cuda")
    smp = torch.zeros(tc, dtype=torch.int32, device="cuda")
    c.collect_device(None, smp.data_ptr(), db.data_ptr())
    cap = c.csv_capacity(tc, len(STAMP))
    text = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    n = torch.zeros(1, dtype=torch.int64, device="cuda")
    c.format_csv_device(STAMP, 0, tc, db.data_ptr(), dc, smp.data_ptr(), text.data_ptr(), cap, n.data_ptr())
    c.sync()
    want = want_text(plan, a)
    assert text[: int(n.item())].cpu().numpy().tobytes() == want
    assert b.collect_csv(STAMP) == want
    # a value outside the domain in a caller's buffer: length -1, no text
    db[3, 5] = 1e300
    c.format_csv_device(STAMP, 0, tc, db.data_ptr(), dc, smp.data_ptr(), text.data_ptr(), cap, n.data_ptr())
    c.sync()
    assert int(n.item()) == -1
    # too small a buffer: an error before anything is touched, the accumulators of b are intact
    feed(port_oracle, pd, (a, b), 2, SYNTH_BIASED, 8)
    out = np.zeros(b.csv_capacity(tc, len(STAMP)) - 1, dtype=np.uint8)
    with pytest.raises(ScanError) as e:
        b.collect_csv(STAMP, out=out)
    assert e.value.code == -4
    with pytest.raises(ScanError):
        c.format_csv_device(STAMP, 0, tc, db.data_ptr(), dc, smp.data_ptr(), text.data_ptr(), cap - 1, n.data_ptr())
    assert b.collect_csv(STAMP) == want_text(plan, a)
    for g in (a, b, c):
        g.close()
