"""The CUDA kernel SOURCE (rtlsdr_b200/csrc/*.cuh) compiled with g++ against the
test-only emulator tests/emu/cuda_emu.h and compared with the oracle.  This is
how kernel index math is checked on the GPU-less build box; the -m gpu suite
repeats the same cases on real hardware through the C ABI."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracles import SYNTH_BIASED, SYNTH_CONST, SYNTH_TONE, SYNTH_XORSHIFT
from scan_cases import expected, make_reads, plan_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")
EMU_SO = os.path.join(EMU_DIR, "libscan_emu.so")


def vp(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


@pytest.fixture(scope="module")
def emu():
    srcs = [os.path.join(EMU_DIR, f) for f in ("emu_entry.cpp", "emu_large.inl", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    srcs.append(os.path.join(ROOT, "include", "rtlsdr_gpu_scan.h"))  # scan_host.cuh reads the config struct
    if not os.path.exists(EMU_SO) or any(os.path.getmtime(s) > os.path.getmtime(EMU_SO) for s in srcs):
        subprocess.run(["g++", "-std=c++20", "-O2", "-DSCAN_EMU", "-I" + EMU_DIR, "-I" + CSRC, "-shared",
                        "-fPIC", "-pthread", "-o", EMU_SO, os.path.join(EMU_DIR, "emu_entry.cpp")], check=True)
    return ctypes.CDLL(EMU_SO)


def sort_by_hop(reads, hops, tune_count, split=2):
    order = np.argsort(hops, kind="stable")
    reads, hops = np.ascontiguousarray(reads[order]), hops[order]
    segs = []
    for h in range(tune_count):
        idx = np.nonzero(hops == h)[0]
        if len(idx) == 0:
            continue
        cuts = np.linspace(0, len(idx), min(split, len(idx)) + 1).astype(int)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                segs.append((h, idx[0] + a, b - a, 0))
    return reads, hops, np.array(segs, dtype=np.int32)


@pytest.mark.parametrize("bin_e", list(range(1, 13)))
def test_small_u8_kernel(emu, port_oracle, bin_e):
    n = 1 << bin_e
    rng = np.random.default_rng(bin_e)
    for peak in (0, 1):
        plan = plan_dict(bin_e, peak_hold=peak, tune_count=2)
        win = rng.integers(-70000, 70000, n).astype(np.int32) if bin_e % 2 else port_oracle.window_coefs("hamming", n)
        reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=10)
        reads[1, :] = 255
        reads[2, :] = 0
        want, want_smp, _ = expected(port_oracle, plan, win, reads, hops)
        sreads, shops, _ = sort_by_hop(reads, hops, 2)
        shops = np.ascontiguousarray(shops, dtype=np.int32)
        sine = port_oracle.sine_table(bin_e)
        # the CTAs share the 6 reads in equal runs (cut at whole reads in so short a launch): 1 CTA, uneven
        # runs (4, 5 CTAs), one read per CTA, and more CTAs than reads
        for grid in ((1, 5) if bin_e < 12 else (1, 2, 4, 5, 6, 9)):
            avg = np.zeros((2, n), dtype=np.int64)
            smp = np.zeros(2, dtype=np.int64)
            emu.emu_small_u8(bin_e, peak, vp(sreads), len(sreads), vp(shops), grid, vp(sine), vp(win), vp(avg), vp(smp))
            assert np.array_equal(avg, want), (bin_e, peak, grid)
            assert np.array_equal(smp, want_smp), (bin_e, peak, grid)


@pytest.mark.parametrize("bin_e,peak", [(12, 0), (10, 1), (7, 0)])
def test_small_u8_kernel_half_read_cuts(emu, port_oracle, bin_e, peak):
    """launches with >= 4 reads per CTA are cut at half reads: 9 reads of 3 hops on 2 CTAs = 9 working sets
    each, the cut falls in the middle of read 4 (both CTAs stage it and take its DC term, each transforms
    its half); the first CTA's run covers a hop boundary, the second starts mid-hop"""
    n = 1 << bin_e
    plan = plan_dict(bin_e, peak_hold=peak, tune_count=3)
    win = port_oracle.window_coefs("blackman", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=40 + bin_e, param=-12)
    reads[4, ::3] = 255
    want, want_smp, _ = expected(port_oracle, plan, win, reads, hops)
    sreads, shops, _ = sort_by_hop(reads, hops, 3)
    shops = np.ascontiguousarray(shops, dtype=np.int32)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((3, n), dtype=np.int64)
    smp = np.zeros(3, dtype=np.int64)
    emu.emu_small_u8(bin_e, peak, vp(sreads), len(sreads), vp(shops), 2, vp(sine), vp(win), vp(avg), vp(smp))
    assert np.array_equal(avg, want)
    assert np.array_equal(smp, want_smp)


@pytest.mark.parametrize("freq,window,fir,peak", [
    ("100M:100.1M:100", "rectangle", -1, 0), ("100M:100.1M:100", "blackman", 9, 0),
    ("100M:100.1M:100", "youssef", 0, 1), ("100M:100.5M:10k", "bartlett", -1, 0),
    ("100M:100.3M:3k", "hamming", -1, 1), ("100M:100.9M:30k", "hamming", -1, 0),
    ("100M:100.01M:50", "hamming", 9, 0),
    ("100M:100.02M:100", "hamming", -1, 0),    # boxcar ds=140: thread-per-slot kernel, 16-byte loads
    ("100M:100.03M:100", "blackman", -1, 1)])  # boxcar ds=93
def test_decimating_kernels(emu, port_oracle, freq, window, fir, peak):
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(freq, 0.0, None if fir < 0 else fir).as_dict()
    plan["peak_hold"] = peak
    bin_e, n = plan["bin_e"], 1 << plan["bin_e"]
    win = port_oracle.window_coefs(window, n)
    for mode, param in ((SYNTH_XORSHIFT, 0), (SYNTH_BIASED, 40), (SYNTH_CONST, 255), (SYNTH_TONE, 127)):
        reads, hops = make_reads(port_oracle.lib, plan, 2, mode, seed=3, param=param)
        want, _, _ = expected(port_oracle, plan, win, reads, hops)
        segs = np.array([(0, 0, len(reads), 0)], dtype=np.int32)
        sine = port_oracle.sine_table(bin_e)
        avg = np.zeros((1, n), dtype=np.int64)
        box = plan["boxcar"] and plan["downsample"] > 1
        fir5 = None
        if not box and plan["comp_fir_size"] == 9 and plan["downsample_passes"] <= 10:
            fir5 = np.array(list(port_oracle.lib.oracle_cic9(plan["downsample_passes"]).contents)[1:6], dtype=np.int32)
        emu.emu_small_decim(bin_e, peak, vp(reads), len(reads), plan["buf_len"], plan["downsample"],
                            plan["downsample_passes"], 0 if box else 1, vp(fir5), vp(segs), 1, vp(sine), vp(win),
                            vp(avg), None, None)
        assert np.array_equal(avg, want), (freq, mode)


@pytest.mark.parametrize("bin_e,peak", [(13, 0), (13, 1), (14, 0), (15, 0), (16, 1), (17, 0), (18, 1)])
def test_large_kernels(emu, port_oracle, bin_e, peak):
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=2 * n, peak_hold=peak, tune_count=2)
    win = port_oracle.window_coefs("blackman-harris" if bin_e % 2 else "hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=bin_e, param=35)
    reads, hops = reads[:3], hops[:3]
    want, _, _ = expected(port_oracle, plan, win, reads, hops)
    sreads, shops, _ = sort_by_hop(reads, hops, 2)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((2, n), dtype=np.int64)
    # pipelined round B (the default for N >= 2^17) and the one-tile-per-CTA kernel it replaces (A/B switch)
    for pipe in (1, 0):
        avg[:] = 0
        emu.emu_set_large_pipe(pipe)
        emu.emu_large(bin_e, peak, 0, vp(sreads), len(sreads), vp(shops.astype(np.int32)), vp(sine), vp(win), None, vp(avg))
        assert np.array_equal(avg, want), pipe
    emu.emu_set_large_pipe(1)


def test_rms_and_epilogue_kernels(emu, port_oracle):
    rng = np.random.default_rng(3)
    for peak in (0, 1):
        plan = plan_dict(0, tune_count=3, peak_hold=peak, rate=1000000)
        reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=1, param=50)
        want, smp, db = expected(port_oracle, plan, np.zeros(1, np.int32), reads, hops)
        for warp_kernel in (0, 1):          # CTA-per-read (default for 16384-byte reads) and warp-per-read kernels
            emu.emu_set_rms_warp(warp_kernel)
            avg = np.zeros(3, dtype=np.int64)
            emu.emu_rms(vp(reads), len(reads), 16384, vp(hops.astype(np.int32)), peak, vp(avg))
            assert np.array_equal(avg, want[:, 0]), warp_kernel
        emu.emu_set_rms_warp(0)
        out = np.zeros((3, 2), dtype=np.float64)
        emu.emu_epilogue(vp(avg), vp(smp.astype(np.int32)), vp(out), 0, 0, 0, 1000000, 3)
        assert np.allclose(out, db, rtol=1e-12)
    # dB epilogue with crop on a 256-bin spectrum, incl. a zero bin (-inf)
    avg = rng.integers(1, 1 << 40, (2, 256)).astype(np.int64)
    avg[1, 7] = 0
    smp = np.array([8, 24], dtype=np.int32)
    crop = 0.3
    i1, i2 = int(256 * crop * 0.5), 255 - int(256 * crop * 0.5)
    out = np.zeros((2, i2 - i1 + 2), dtype=np.float64)
    emu.emu_epilogue(vp(avg), vp(smp), vp(out), 8, i1, i2, 2400000, 2)
    for h in range(2):
        _, db = port_oracle.epilogue(avg[h], 8, crop, 2400000, int(smp[h]))
        fin = np.isfinite(db)
        assert np.array_equal(np.isfinite(out[h]), fin)
        assert np.allclose(out[h][fin], db[fin], rtol=1e-12)


@pytest.mark.parametrize("bin_e,ds", [(1, 7), (2, 3), (3, 5), (4, 2), (6, 11), (12, 2)])
def test_decimating_small_n_multi_segment(emu, port_oracle, bin_e, ds):
    """boxcar images of consecutive reads are packed back to back: FFT blocks of several
    reads share a working set (and, for N < 16, a thread); two hops, uneven segments."""
    n = 1 << bin_e
    buf_len = max(16384, 2 * n * ds)
    plan = plan_dict(bin_e, buf_len=buf_len, downsample=ds, tune_count=2, peak_hold=bin_e % 2)
    win = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=45)
    reads, hops = reads[:5], hops[:5]
    want, _, _ = expected(port_oracle, plan, win, reads, hops)
    sreads, shops, segs = sort_by_hop(reads, hops, 2, split=2)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((2, n), dtype=np.int64)
    emu.emu_small_decim(bin_e, plan["peak_hold"], vp(sreads), len(sreads), buf_len, ds, 0, 0, None, vp(segs),
                        len(segs), vp(sine), vp(win), vp(avg), None, None)
    assert np.array_equal(avg, want)


@pytest.mark.parametrize("passes,fir", [(1, 9), (2, 0), (3, 9), (4, 5), (5, 9), (6, 9), (7, 9), (8, 9)])
def test_fifth_order_chain_every_depth(emu, port_oracle, passes, fir):
    """fused fifth_order x P (+ FIR) tile kernel for P <= 7, per-pass kernels beyond"""
    bin_e = 6
    n, ds = 1 << bin_e, 1 << passes
    buf_len = max(16384, 2 * n * ds)
    plan = plan_dict(bin_e, buf_len=buf_len, downsample=ds, downsample_passes=passes, boxcar=0,
                     comp_fir_size=fir, tune_count=1)
    win = port_oracle.window_coefs("blackman", n)
    reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=passes, param=30)
    reads[1, 100:300] = 255
    want, _, _ = expected(port_oracle, plan, win, reads, hops)
    segs = np.array([(0, 0, 2, 0)], dtype=np.int32)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((1, n), dtype=np.int64)
    fir5 = None
    if fir == 9 and passes <= 10:
        fir5 = np.array(list(port_oracle.lib.oracle_cic9(passes).contents)[1:6], dtype=np.int32)
    emu.emu_small_decim(bin_e, 0, vp(reads), 2, buf_len, ds, passes, 1, vp(fir5), vp(segs), 1, vp(sine), vp(win),
                        vp(avg), None, None)
    assert np.array_equal(avg, want)


def test_level_stats_kernel(emu):
    rng = np.random.default_rng(4)
    reads = rng.integers(0, 256, (9, 16384), dtype=np.uint8)
    reads[2, :5000] = 255
    reads[5, 100:900] = 0
    hop_of = np.array([0, 1, 2, 0, 1, 2, 0, 1, 2], dtype=np.int32)
    level = np.zeros((3, 2), dtype=np.uint64)
    emu.emu_level_stats(vp(reads), 9, 16384, vp(hop_of), vp(level))
    for h in range(3):
        b = reads[hop_of == h]
        assert level[h, 0] == np.count_nonzero((b == 0) | (b == 255))     # librtlsdr.c:3302
        assert level[h, 1] == np.count_nonzero((b < 64) | (b > 191))      # librtlsdr.c:3304


@pytest.mark.parametrize("bin_e,ds,slots", [(8, 2, 2), (8, 13, 3), (9, 28, 12), (10, 28, 6), (10, 64, 2), (11, 5, 4), (12, 3, 3)])
def test_fused_boxcar_kernel(emu, port_oracle, bin_e, ds, slots):
    """boxcar + DC + window + FFT + |X|^2 in one kernel (narrow scans, one FFT block per read)"""
    n = 1 << bin_e
    buf_len = 2 * n * ds
    for peak in (0, 1):
        plan = plan_dict(bin_e, buf_len=buf_len, downsample=ds, tune_count=2, peak_hold=peak)
        win = port_oracle.window_coefs("blackman", n)
        reads, hops = make_reads(port_oracle.lib, plan, 5, SYNTH_BIASED, seed=bin_e + ds, param=35)
        reads, hops = reads[:9], hops[:9]
        reads[3, :] = 255
        want, want_smp, _ = expected(port_oracle, plan, win, reads, hops)
        sreads, _, segs = sort_by_hop(reads, hops, 2, split=2)
        sine = port_oracle.sine_table(bin_e)
        avg = np.zeros((2, n), dtype=np.int64)
        smp = np.zeros(2, dtype=np.int64)
        emu.emu_fused_boxcar(bin_e, peak, vp(sreads), len(sreads), ds, slots, vp(segs), len(segs), vp(sine), vp(win),
                             vp(avg), vp(smp))
        assert np.array_equal(avg, want), (bin_e, ds, peak)
        assert np.array_equal(smp, want_smp)


@pytest.mark.parametrize("bin_e,ds,slots,grid", [(8, 2, 3, 1), (8, 13, 16, 2), (9, 28, 5, 3), (10, 28, 10, 2), (10, 64, 3, 1),
                                                 (11, 5, 4, 2), (12, 3, 3, 2), (12, 12, 8, 1)])
@pytest.mark.parametrize("mode", [1, 2, 3, 5])
def test_stream_boxcar_kernel(emu, port_oracle, bin_e, ds, slots, grid, mode):
    """warp-specialised narrow-scan kernel: bulk-copy producer, boxcar warps, transform warps (mbarrier hand-offs)"""
    n = 1 << bin_e
    buf_len = 2 * n * ds
    for peak in (0, 1):
        plan = plan_dict(bin_e, buf_len=buf_len, downsample=ds, tune_count=2, peak_hold=peak)
        win = port_oracle.window_coefs("blackman", n)
        passes = 5 if n * ds > 4096 else 40   # small reads: several working sets per segment
        reads, hops = make_reads(port_oracle.lib, plan, passes, SYNTH_BIASED, seed=bin_e + ds, param=35)
        reads, hops = reads[:2 * passes - 1], hops[:2 * passes - 1]
        reads[3, :] = 255
        want, want_smp, _ = expected(port_oracle, plan, win, reads, hops)
        sreads, _, segs = sort_by_hop(reads, hops, 2, split=2)
        sine = port_oracle.sine_table(bin_e)
        avg = np.zeros((2, n), dtype=np.int64)
        smp = np.zeros(2, dtype=np.int64)
        if mode in (1, 3):
            slots = max(4, slots & ~1)   # two boxcar groups: even ring, a slot always serves the same group
        emu.emu_stream_boxcar(bin_e, peak, mode, vp(sreads), len(sreads), ds, slots, grid, vp(segs), len(segs), vp(sine), vp(win),
                              vp(avg), vp(smp))
        assert np.array_equal(avg, want), (bin_e, ds, peak)
        assert np.array_equal(smp, want_smp)


@pytest.mark.parametrize("passes,fir,span", [(1, 9, 64), (1, 0, 4096), (2, 9, 256), (3, 9, 64), (3, 0, 1024), (4, 9, 128),
                                             (4, 5, 512), (5, 9, 64), (5, 0, 256)])
def test_fifth_order_streaming_kernel(emu, port_oracle, passes, fir, span):
    """register-streaming -F chain (levels in registers, level 1 straight from the bytes) + 16-sample head tiles"""
    bin_e = 6
    n, ds = 1 << bin_e, 1 << passes
    buf_len = max(16384, 2 * n * ds)
    plan = plan_dict(bin_e, buf_len=buf_len, downsample=ds, downsample_passes=passes, boxcar=0,
                     comp_fir_size=fir, tune_count=1)
    win = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=40 + passes, param=-45)
    reads[1, 100:300] = 255
    reads[2, :64] = 0
    reads[2, 5000:5100] = 255
    want, _, _ = expected(port_oracle, plan, win, reads, hops)
    segs = np.array([(0, 0, 3, 0)], dtype=np.int32)
    sine = port_oracle.sine_table(bin_e)
    avg = np.zeros((1, n), dtype=np.int64)
    fir5 = None
    if fir == 9:
        fir5 = np.array(list(port_oracle.lib.oracle_cic9(passes).contents)[1:6], dtype=np.int32)
    emu.emu_set_hb_span(span)
    emu.emu_small_decim(bin_e, 0, vp(reads), 3, buf_len, ds, passes, 2, vp(fir5), vp(segs), 1, vp(sine), vp(win),
                        vp(avg), None, None)
    assert np.array_equal(avg, want)
