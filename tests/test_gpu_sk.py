"""Spectral kurtosis on the GPU (RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS): twin handles with the flag on and off get
the same bytes; S2 equals the oracle's 128-bit sums; the SK rows equal sk.cuh's host evaluation bit for bit; the
estimator behaves (noise ~ 1, intermittent tone > 1, steady tone < 1); rtl_power_gpu -K."""
import os
import subprocess

import numpy as np
import pytest

from oracles import SYNTH_BIASED, SYNTH_XORSHIFT
from scan_cases import make_reads, plan_dict
from test_sk import expected_sk_rows, full_scale, oracle_sk, same_bits, sk_emu  # noqa: F401  (sk_emu: fixture)

pytestmark = pytest.mark.gpu
STAMP = "2026-01-01, 00:00:00, "


@pytest.fixture(scope="module")
def scan_mod():
    import rtlsdr_b200.scan as s
    s.load_library()
    return s


def host_sk_rows(sk_emu, avg, smp, s2, pd):
    """expected_sk_rows() through the host build of sk_from_moments (the library's header, compiled by g++)"""
    f = lambda s1, S2, m: sk_emu.emu_sk_from_moments(s1, S2 & ((1 << 64) - 1), S2 >> 64, m)  # noqa: E731
    want, _, _ = expected_sk_rows(avg, smp, s2, pd["bin_e"], pd["crop"], pd["downsample"], f)
    return want


def feed(handles, pd, reads, hops, how, scan_mod):
    tc, b = pd["tune_count"], pd["buf_len"]
    if how == "submit":
        for g in handles:
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
        return
    passes = len(reads) // tc
    assert np.array_equal(hops, np.tile(np.arange(tc), passes))
    if how == "batch":
        pinned = scan_mod.PinnedBuffer(reads.nbytes)
        pinned.array[:] = reads.reshape(-1)
        for g in handles:
            g.submit_batch(0, tc, passes, pinned.ptr, tc * b, b)
            g.sync()
        return
    import torch
    dev = torch.from_numpy(np.ascontiguousarray(reads)).cuda()
    torch.cuda.synchronize()
    for g in handles:
        g.submit_device(0, tc, passes, dev.data_ptr(), tc * b, b)
        g.sync()


def check_report(scan_mod, sk_emu, port_oracle, pd, w, a, b, reads, hops):
    avg, smp, db = a.collect_all()
    avg2, smp2, db2, s2, sk = b.collect_sk()
    assert avg.tobytes() == avg2.tobytes() and smp.tobytes() == smp2.tobytes() and db.tobytes() == db2.tobytes()
    want_avg, want_smp, want_s2 = oracle_sk(port_oracle, pd, w, reads, hops)
    assert np.array_equal(avg, want_avg) and np.array_equal(smp, want_smp)
    assert np.array_equal(s2, want_s2)
    want = host_sk_rows(sk_emu, avg, smp, s2, pd)
    assert all(same_bits(x, y) for x, y in zip(sk.ravel(), want.ravel()))
    return s2, sk


def twins(scan_mod, pd, w, **kw):
    a = scan_mod.GpuScan.from_plan(pd, window_coefs=w, **kw)
    b = scan_mod.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True, **kw)
    return a, b


@pytest.mark.parametrize("bin_e,window,how", [(1, "hamming", "submit"), (4, "rectangle", "batch"),
                                              (10, "blackman-harris", "device"), (12, "hamming", "submit"),
                                              (13, "hamming", "device"), (16, "blackman-harris", "batch"),
                                              (17, "hamming", "device")])
def test_sk_twins_three_reports(scan_mod, sk_emu, port_oracle, bin_e, window, how):
    """several hops, three reports (read-and-zero of S2), every submit route; the second report has a
    full-scale read in every hop (S2 carries into the high word), the third constant-127 input (S1 = 0: NaN)"""
    n = 1 << bin_e
    pd = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=3, crop=0.2 if bin_e % 2 else 0.0)
    w = port_oracle.window_coefs(window, n)
    a, b = twins(scan_mod, pd, w)
    try:
        for rep in range(3):
            reads, hops = make_reads(port_oracle.lib, pd, 2, SYNTH_BIASED, seed=10 * bin_e + rep, param=25)
            if rep == 1:
                reads[:3] = full_scale(pd["buf_len"])
            if rep == 2:
                reads[:] = 127
            feed((a, b), pd, reads, hops, how, scan_mod)
            s2, sk = check_report(scan_mod, sk_emu, port_oracle, pd, w, a, b, reads, hops)
            if rep == 1 and window == "rectangle":
                assert s2[..., 1].any()   # 512 full-scale blocks per hop
            if rep == 2:
                assert not s2.any() and np.isnan(sk).all()
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("freq,fir", [("100M:100.1M:100", None), ("100M:100.3M:3k", 9)])
def test_sk_decimating_scans(scan_mod, sk_emu, port_oracle, freq, fir):
    """narrow boxcar ds = 28 at 1024 bins (the staged route instead of the warp-specialised kernels) and -F 9"""
    from rtlsdr_b200.planner import plan_scan
    pd = plan_scan(freq, 0.0 if fir is None else 0.1, fir).as_dict()
    pd["peak_hold"] = 0
    if fir is None:
        assert pd["downsample"] == 28 and pd["bin_e"] == 10
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    a, b = twins(scan_mod, pd, w)
    try:
        for rep in range(2):
            reads, hops = make_reads(port_oracle.lib, pd, 6, SYNTH_XORSHIFT, seed=rep)
            reads[1] = full_scale(pd["buf_len"])
            feed((a, b), pd, reads, hops, "device" if rep else "submit", scan_mod)
            check_report(scan_mod, sk_emu, port_oracle, pd, w, a, b, reads, hops)
    finally:
        a.close()
        b.close()


def test_sk_csv_text_unchanged(scan_mod, port_oracle):
    """collect_csv of an SK handle prints the same bytes as without the flag, and zeroes S2"""
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan("88M:108M:25k", 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    a, b = twins(scan_mod, pd, w)
    try:
        a.set_csv_columns(*plan.csv_columns())
        b.set_csv_columns(*plan.csv_columns())
        reads, hops = make_reads(port_oracle.lib, pd, 3, SYNTH_BIASED, seed=4, param=30)
        feed((a, b), pd, reads, hops, "submit", scan_mod)
        assert a.collect_csv(STAMP) == b.collect_csv(STAMP)
        _, smp, _, s2, sk = b.collect_sk()
        assert not smp.any() and not s2.any() and np.isnan(sk).all()
    finally:
        a.close()
        b.close()


def tone_reads(rng, n_reads, n, k0, amp, on):
    """uniform noise bytes plus, in the reads where on[i], a complex tone exactly on bin k0 of an n-point block"""
    t = np.arange(8192)
    reads = rng.integers(127 - 60, 128 + 60, (n_reads, 16384)).astype(np.float64)
    for i in range(n_reads):
        if on[i]:
            ph = 2 * np.pi * k0 * t / n + rng.uniform(0, 2 * np.pi)
            reads[i, 0::2] += amp * np.cos(ph)
            reads[i, 1::2] += amp * np.sin(ph)
    return np.clip(np.round(reads), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("bin_e", [5, 6])
def test_sk_statistics(scan_mod, bin_e):
    """noise: mean SK ~ 1; a tone in a quarter of the reads: SK > 2 (ideal 1/p - 1 = 3); a steady tone: SK < 0.5.
    (Only small transforms: fix_fft halves at every stage, so larger ones quantise noise to about one LSB.)"""
    n, k0 = 1 << bin_e, 5
    cols = [(k0 + n // 2) % n, (n - k0 + n // 2) % n]   # the tone's column in the half-swapped row, either sign
    rng = np.random.default_rng(bin_e)
    g = scan_mod.GpuScan(1, bin_e, 16384, spectral_kurtosis=True)
    try:
        noise = rng.integers(0, 256, (16, 16384), dtype=np.uint8)
        for r in noise:
            g.submit(0, r)
        sk = g.collect_sk()[4][0]
        assert abs(np.mean(sk) - 1.0) < 0.05, np.mean(sk)
        for on, check in (([i % 4 == 0 for i in range(16)], lambda v: max(v) > 2.0), ([True] * 16, lambda v: min(v) < 0.5)):
            for r in tone_reads(rng, 16, n, k0, 60.0, on):
                g.submit(0, r)
            sk = g.collect_sk()[4][0]
            assert check(sk[cols]), (sk[cols], on[:4])
    finally:
        g.close()


def test_sk_rejects_device_report_and_merge(scan_mod):
    import torch
    g = scan_mod.GpuScan(2, 10, 16384, spectral_kurtosis=True)
    try:
        d_avg = torch.zeros((2, 1024), dtype=torch.int64, device="cuda")
        d_smp = torch.zeros(2, dtype=torch.int32, device="cuda")
        d_db = torch.zeros((2, g.db_count), dtype=torch.float64, device="cuda")
        with pytest.raises(scan_mod.ScanError) as e:
            g.collect_device(d_avg.data_ptr(), d_smp.data_ptr(), d_db.data_ptr())
        assert e.value.code == -2
        with pytest.raises(scan_mod.ScanError) as e:
            g.merge_device(d_avg.data_ptr(), d_smp.data_ptr())
        assert e.value.code == -2
    finally:
        g.close()
    plain = scan_mod.GpuScan(2, 10, 16384)
    try:
        with pytest.raises(scan_mod.ScanError) as e:
            plain.collect_sk()
        assert e.value.code == -2
    finally:
        plain.close()


def test_cli_sk_file(scan_mod, port_oracle, tmp_path):
    """rtl_power_gpu -K: rows with the power rows' prefix, values %.4f of collect_sk (nan where undefined);
    -K with more workers than hops is refused"""
    from rtlsdr_b200 import _build
    from rtlsdr_b200.planner import plan_scan
    _build.build_host()
    exe = os.path.join(_build.HOST_BUILD, "rtl_power_gpu")
    out, skf = tmp_path / "scan.csv", tmp_path / "sk.csv"
    env = dict(os.environ, RTLSDR_SYNTH_MODE="biased", RTLSDR_SYNTH_SEED="3", RTLSDR_SYNTH_PARAM="21",
               RTL_POWER_PASSES="4", RTL_POWER_TIMESTAMP="2026-01-01, 00:00:00")
    r = subprocess.run([exe, "-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "-1", "-K", str(skf), str(out)],
                       env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    plan = plan_scan("88M:108M:25k", 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    reads, hops = make_reads(port_oracle.lib, pd, 4, SYNTH_BIASED, seed=3, param=21)
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True)
    rows, sk_rows = [], []
    try:
        for rd, h in zip(reads, hops):
            g.submit(int(h), rd)
        _, smp, db, _, sk = g.collect_sk()
        for h in range(pd["tune_count"]):
            rows.append(STAMP + plan.csv_row(h, int(smp[h]), db[h]))
            prefix = rows[-1].split(", ")[:6]
            vals = ["nan" if v != v else "%.4f" % v for v in sk[h]]
            sk_rows.append(", ".join(prefix + vals) + "\n")
    finally:
        g.close()
    assert out.read_text() == "".join(rows)
    assert skf.read_text() == "".join(sk_rows)
    r = subprocess.run([exe, "-f", "100M:100.1M:100", "-t", "2", "-K", str(skf), str(out)],
                       env=dict(env, RTLSDR_GPU_DEVICES="0,0"), capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "-K" in r.stderr
