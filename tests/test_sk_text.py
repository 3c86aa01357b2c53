"""Spectral-kurtosis rows and merges on the CPU: the %.4f formatter of rtlsdr_b200/csrc/csv_text.cuh against glibc's
snprintf on >= 10 M values, csv_sk_rows_kernel against the bytes rtl_power_gpu -K has always written,
merge_sk_sets_kernel (sk.cuh) against Python integer sums with carries chained across sets (all through
tests/emu/sk_text_entry.cpp and the CPU emulator), and SpectrumGather(sk=True)'s slot layout over world-2 gloo."""
import ctypes
import math
import os
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")
STAMP = "2026-01-01, 00:00:00, "
ROW_FIXED, SK_VALUE_MAX = 56, 17
U64 = (1 << 64) - 1


def vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sk_text_emu") / "libsk_text_emu.so")
    subprocess.run(["g++", "-std=c++20", "-O2", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC, "-shared", "-fPIC",
                    "-pthread", "-o", so, os.path.join(EMU_DIR, "sk_text_entry.cpp")], check=True)
    L = ctypes.CDLL(so)
    i64, p, i = ctypes.c_longlong, ctypes.c_void_p, ctypes.c_int
    L.emu_csv_check_f4.argtypes = [p, i64, ctypes.POINTER(i64)]
    L.emu_csv_check_f4.restype = i64
    L.emu_csv_f4.argtypes = [ctypes.c_double, ctypes.c_char_p]
    L.emu_sk_csv_rows.argtypes = [ctypes.c_char_p, i, i, p, i64, p, p, p, i, ctypes.c_double, i, p]
    L.emu_sk_csv_rows.restype = i64
    L.emu_merge_sk.argtypes = [p, p, p, p, p, p, i64, i64, i, i, i]
    L.emu_merge_sk.restype = None
    return L


def f4_values(rng):
    """every class of double the %.4f formatter is specified for"""
    top = 2.0 ** 53
    parts = [rng.uniform(0, 2.0 ** 31 + 2, 4_000_000),                       # SK values up to M + 1, M < 2^31
             rng.uniform(0, 4, 2_000_000),                                   # SK near 1
             np.arange(-100_000, 100_000, dtype=np.float64),                 # integers
             rng.integers(-(1 << 53) + 1, 1 << 53, 200_000).astype(np.float64)]
    # exact ties between two 4-decimal values: odd multiples of 2^-k that are also multiples of 10^-4 / 2 = 2^-5 * ...
    k = np.arange(1, 400_001, dtype=np.float64)
    parts += [(2 * k - 1) / 32.0, (2 * k - 1) / 32.0 + 1.0, -(2 * k - 1) / 32.0, (2 * k - 1) / 2.0 ** 5 * 3]
    bound = (np.arange(-300_000, 300_000) + 0.5) / 10_000.0                  # rounding boundaries (j + 1/2) / 10^4
    parts += [bound, np.nextafter(bound, np.inf), np.nextafter(bound, -np.inf)]
    # random bit patterns below 2^53: any sign, mantissa and biased exponent up to 1075
    bits = rng.integers(0, 1 << 52, 2_000_000, dtype=np.uint64)
    bits |= rng.integers(0, 1076, 2_000_000, dtype=np.uint64) << np.uint64(52)
    bits |= rng.integers(0, 2, 2_000_000, dtype=np.uint64) << np.uint64(63)
    parts.append(bits.view(np.float64))
    parts.append(-rng.uniform(0, 1e-4, 300_000))                             # tiny negatives: -0.0000 / -0.0001
    sub = rng.integers(1, 1 << 52, 300_000, dtype=np.uint64)                 # subnormals of both signs
    sub[::2] |= np.uint64(1) << np.uint64(63)
    parts.append(sub.view(np.float64))
    parts.append(np.array([0.0, -0.0, np.inf, -np.inf, np.nextafter(top, 0), -np.nextafter(top, 0), 5e-324, -5e-324,
                           0.03125, 1.21875, 0.00005, -0.00005, 0.00015, 0.99995, 9.99995, 2147483649.0,
                           2.0 ** 31 + 1 - 2.0 ** -21, 1 - 2.0 ** -53, 2.0 ** -14, 2.0 ** -15, 2.0 ** -67,
                           2.0 ** -66 * 3, 2.0 ** 52 + 0.5, 2.0 ** 52 - 0.5]))
    nan_bits = np.array([0x7FF0000000000001, 0x7FF8000000000000, 0xFFF8000000000000, 0xFFFFFFFFFFFFFFFF,
                         0xFFF0000000000001], dtype=np.uint64)
    parts.append(nan_bits.view(np.float64))
    return np.ascontiguousarray(np.concatenate(parts))


def test_f4_matches_printf(emu):
    v = f4_values(np.random.default_rng(5))
    assert v.size >= 10_000_000
    first = ctypes.c_longlong()
    bad = emu.emu_csv_check_f4(vp(v), v.size, ctypes.byref(first))
    assert bad == 0, f"{bad} mismatches, first {v[first.value]!r}"


def test_f4_domain_edges(emu):
    buf = ctypes.create_string_buffer(32)
    top = 2.0 ** 53
    assert emu.emu_csv_f4(np.nextafter(top, 0), buf) == 21 and buf.value == b"9007199254740991.0000"
    assert emu.emu_csv_f4(-np.nextafter(top, 0), buf) == 22 and buf.value == b"-9007199254740991.0000"
    for x in (top, -top, 1e300, -1.7e308):
        assert emu.emu_csv_f4(x, buf) == -1
    assert emu.emu_csv_f4(-0.0, buf) == 7 and buf.value == b"-0.0000"
    assert emu.emu_csv_f4(-1e-300, buf) == 7 and buf.value == b"-0.0000"
    assert emu.emu_csv_f4(0.03125, buf) == 6 and buf.value == b"0.0312"      # tie, to even
    assert emu.emu_csv_f4(1.21875, buf) == 6 and buf.value == b"1.2188"      # tie, to even
    for nan in (np.nan, -np.nan):
        assert emu.emu_csv_f4(nan, buf) == 3 and buf.value == b"nan"


def sk_row_text(stamp, low, high, step, smp, vals):
    """the bytes rtl_power_gpu -K has written for one SK row (host printf: power row prefix, %.4f, nan)"""
    head = "%s%i, %i, %.2f, %i, " % (stamp, low, high, step, smp)
    return head + ", ".join("nan" if math.isnan(v) else "%.4f" % v for v in vals) + "\n"


def emu_sk_rows(emu, low, high, step, row_first, rows, sk, smp, stamp=STAMP):
    cap = rows * (len(stamp) + ROW_FIXED + SK_VALUE_MAX * sk.shape[1])
    text = np.zeros(cap, dtype=np.uint8)
    n = emu.emu_sk_csv_rows(stamp.encode(), row_first, rows, vp(sk), sk.shape[1], vp(smp), vp(low), vp(high),
                            low.size, step, sk.shape[1], vp(text))
    return n, text


@pytest.mark.parametrize("rng_,crop", [("88M:108M:1M", 0.2), ("100M:102M:2.5k", 0.0), ("88M:108M:1k", 0.2),
                                       ("100M:101M:10", 0.0)])
def test_sk_row_kernels_match_host_rows(emu, rng_, crop):
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(rng_, crop)
    rng = np.random.default_rng(plan.bin_e)
    low, high, step = plan.csv_columns()
    row_first = 1 if plan.tune_count > 3 else 0
    rows = min(plan.tune_count - row_first, 3)
    sk = rng.uniform(0, 3, (rows, plan.db_count))
    sk[:, rng.integers(0, plan.db_count, max(1, plan.db_count // 20))] = np.nan
    sk[0, 0] = -np.nan
    sk[0, -1] = -1e-17                                   # rounding below c = 1: -0.0000
    sk[-1, :2] = [2147483649.0, 0.0]
    smp = rng.integers(0, 1 << 20, rows).astype(np.int32)
    n, text = emu_sk_rows(emu, low, high, step, row_first, rows, np.ascontiguousarray(sk), smp)
    want = "".join(sk_row_text(STAMP, low[row_first + r], high[row_first + r], step, smp[r], sk[r])
                   for r in range(rows))
    assert n == len(want)
    assert text[:n].tobytes().decode() == want


def test_sk_capacity_is_tight_for_the_widest_row(emu):
    """the longest SK row: INT32_MIN edges and count, the widest step, every value "2147483649.0000" """
    sk = np.full((1, 3), 2147483649.0)
    smp = np.array([-2 ** 31], dtype=np.int32)
    low = high = smp
    step = np.nextafter(2.0 ** 31, 0)
    n, text = emu_sk_rows(emu, low, high, step, 0, 1, sk, smp)
    cap = len(STAMP) + ROW_FIXED + SK_VALUE_MAX * 3
    want = sk_row_text(STAMP, low[0], high[0], step, smp[0], sk[0])
    assert len(want) <= cap and cap - len(want) <= 3
    assert n == len(want) and text[:n].tobytes().decode() == want
    for bad in (1e10, -1e9, 2.0 ** 53):                  # wider than 15 characters, or outside the domain
        sk[0, 1] = bad
        assert emu_sk_rows(emu, low, high, step, 0, 1, sk, smp)[0] == -1


@pytest.mark.parametrize("own", [False, True])
@pytest.mark.parametrize("bins,hops,sets,grid", [(1024, 1, 3, 4), (3 * 4096, 3, 4, 2), (700, 7, 1, 1)])
def test_merge_sk_sets_kernel(emu, bins, hops, sets, grid, own):
    """S2 low words just below 2^64 in every set, so carries chain across sets; S1 and counts summed too"""
    rng = np.random.default_rng(bins + sets)
    words = bins + bins * 2 + (hops + 1) // 2 + 3         # one padded set: S1, S2, counts
    ext = np.zeros((sets, words), dtype=np.uint64)
    s1 = rng.integers(0, 1 << 50, (sets, bins)).astype(np.int64)
    lo = (np.uint64(U64) - rng.integers(0, 1 << 20, (sets, bins)).astype(np.uint64))
    hi = rng.integers(0, 1 << 40, (sets, bins)).astype(np.uint64)
    cnt = rng.integers(0, 1 << 24, (sets, hops)).astype(np.int32)
    ext[:, :bins] = s1.view(np.uint64)
    ext[:, bins: 3 * bins: 2] = lo
    ext[:, bins + 1: 3 * bins: 2] = hi
    ext[:, 3 * bins: 3 * bins + (hops + 1) // 2].view(np.int32)[:, :hops] = cnt
    if own:
        avg = rng.integers(0, 1 << 50, bins).astype(np.int64)
        smp = rng.integers(0, 1 << 30, hops).astype(np.int64)
        s2 = np.stack([np.full(bins, U64 - 5, dtype=np.uint64), rng.integers(0, 9, bins).astype(np.uint64)], 1)
    else:
        avg, smp, s2 = np.zeros(bins, np.int64), np.zeros(hops, np.int64), np.zeros((bins, 2), np.uint64)
    want_avg = avg + s1.sum(0)
    want_smp = smp + cnt.astype(np.int64).sum(0)
    want_s2 = [int(s2[i, 0]) + (int(s2[i, 1]) << 64) + sum(int(lo[s, i]) + (int(hi[s, i]) << 64) for s in range(sets))
               for i in range(bins)]
    s2 = np.ascontiguousarray(s2)
    base = ext.ctypes.data
    emu.emu_merge_sk(vp(avg), vp(smp), vp(s2), base, base + 3 * bins * 8, base + bins * 8, words * 8, bins, hops,
                     sets, grid)
    assert np.array_equal(avg, want_avg) and np.array_equal(smp, want_smp)
    assert [int(a) + (int(b) << 64) for a, b in s2] == [w & ((1 << 128) - 1) for w in want_s2]
    if sets + own > 1:
        assert all(w >> 64 > int(hi[:, i].sum()) for i, w in enumerate(want_s2))  # carries did happen


# ---- SpectrumGather(sk=True) over gloo --------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_data(tc, n, dbc, r, j):
    """what rank r reports for interval j: deterministic, different per rank, interval and section"""
    rng = np.random.default_rng(1000 * j + r)
    return (rng.integers(0, 1 << 60, (tc, n)).astype(np.int64), rng.uniform(-100, 100, (tc, dbc)),
            rng.integers(0, 1 << 30, tc).astype(np.int32), rng.integers(0, 1 << 63, (tc, n, 2)).astype(np.uint64),
            rng.uniform(0, 3, (tc, dbc)))


def _gather_worker(rank, world, port, tc, n, dbc, replicated, out_path):
    from rtlsdr_b200.sweep import SpectrumGather
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = SpectrumGather(tc, n, dbc, world, rank, "cpu", replicated=replicated, sk=True)
        plain = SpectrumGather(tc, n, dbc, world, rank, "cpu", replicated=replicated)
        ok = plain.words < g.words and g.s2_at == plain.words and g.sk_at == g.s2_at + g.hmax * n * 2
        ok = ok and g.words == g.sk_at + g.hmax * dbc
        for j in range(3):
            k = j & 1
            mine = g.my_hops
            a, d, s, s2, sk = g.views(k)
            data = _rank_data(tc, n, dbc, rank, j)
            for view, src in zip((a, d, s, s2, sk), data):
                view.copy_(torch.from_numpy(np.ascontiguousarray(src[mine.start: mine.stop])))
            g.before_collect(k)
            g.publish(k, to_host=True)
            rep = g.fetch(k)
            if rank == 0:
                raw = g.recv[k].numpy()
                for r in range(world):
                    hops = g.ranges[r]
                    want = _rank_data(tc, n, dbc, r, j)
                    h = len(hops)
                    # the accessor's byte offsets inside a slot hold what rank r wrote
                    b2 = raw[r, g.s2_at: g.s2_at + g.hmax * n * 2].reshape(g.hmax, n, 2)[:h]
                    bk = raw[r, g.sk_at: g.sk_at + g.hmax * dbc].view(np.float64).reshape(g.hmax, dbc)[:h]
                    ok = ok and np.array_equal(b2, want[3][hops.start: hops.stop])
                    ok = ok and np.array_equal(bk, want[4][hops.start: hops.stop])
                    if not replicated:
                        for got, w in zip((rep.avg, rep.db, rep.samples, rep.s2, rep.sk), want):
                            ok = ok and np.array_equal(got[hops.start: hops.stop], w[hops.start: hops.stop])
        if rank == 0:
            with open(out_path, "w") as f:
                f.write("ok" if ok else "mismatch")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("replicated", [False, True])
def test_spectrum_gather_sk_slots_round_trip(tmp_path, replicated):
    out = str(tmp_path / "result")
    mp.spawn(_gather_worker, args=(2, _free_port(), 5, 64, 30, replicated, out), nprocs=2, join=True)
    assert open(out).read() == "ok"
