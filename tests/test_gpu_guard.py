"""Guard-bit transform (RTLSDR_GPU_FLAG_GUARD_BITS) on the GPU: bins and sample counts against the guard oracle
(tests/oracle_guard.c) at every transform path and front end, peak hold, SK, the asynchronous report, short reads,
merged handles, sweep_main --guard-bits and rtl_power_gpu -G; and what the extra bits buy on low-level noise."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracles import SYNTH_BIASED, SYNTH_XORSHIFT
from scan_cases import db_close, make_reads, plan_dict
from test_guard import full_scale, guard_db, oracle_guard
from test_sk import expected_sk_rows, same_bits

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WINDOWS = ["rectangle", "hamming", "blackman", "blackman-harris", "hann-poisson", "youssef", "bartlett"]


@pytest.fixture(scope="module")
def scan_mod():
    import rtlsdr_b200.scan as s
    s.load_library()
    return s


def want_report(plan, avg, smp):
    return np.stack([guard_db(avg[h], plan["bin_e"], plan["crop"], plan["rate"], int(smp[h]))
                     for h in range(avg.shape[0])])


def check_report(got, plan, want_avg, want_smp, what):
    avg, smp, db = got
    assert np.array_equal(avg, want_avg), what
    assert np.array_equal(smp, want_smp), what
    assert db_close(db, want_report(plan, want_avg, want_smp)), what


@pytest.mark.parametrize("bin_e", list(range(1, 15)) + [16, 17, 20, 21])
def test_guard_bins_equal_the_oracle(scan_mod, port_oracle, bin_e):
    """three reports (read-and-zero) through submit, submit_batch and submit_device; several hops"""
    import torch
    n = 1 << bin_e
    tc = 3 if bin_e <= 17 else 2
    plan = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=tc, crop=0.1)
    w = port_oracle.window_coefs(WINDOWS[bin_e % len(WINDOWS)], n)
    g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=True)
    try:
        for rep, route in enumerate(("submit", "batch", "device")):
            reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=bin_e * 3 + rep, param=20)
            if rep == 1:
                reads[0] = full_scale(plan["buf_len"])
            want_avg, want_smp, _ = oracle_guard(port_oracle, plan, w, reads, hops)
            b = plan["buf_len"]
            if route == "submit":
                for r, h in zip(reads, hops):
                    g.submit(int(h), r)
            elif route == "batch":
                buf = scan_mod.PinnedBuffer(reads.size)
                buf.view(np.uint8, reads.shape)[:] = reads
                g.submit_batch(0, tc, 2, buf.ptr, tc * b, b)
                g.sync()
                buf.free()
            else:
                dev = torch.from_numpy(reads).cuda()
                g.submit_device(0, tc, 2, dev.data_ptr(), tc * b, b)
                g.sync()
            check_report(g.collect_all(), plan, want_avg, want_smp, (bin_e, route))
    finally:
        g.close()


LARGE_DECIMATED = {
    # one block of 2^13 / 2^14 points per read behind a boxcar (ds = 4) and behind a -F 9 chain (2 passes, ds = 4)
    "box13": plan_dict(13, buf_len=65536, downsample=4, tune_count=2),
    "fir14": plan_dict(14, buf_len=131072, downsample=4, downsample_passes=2, boxcar=0, comp_fir_size=9, tune_count=2),
}


@pytest.mark.parametrize("freq,fir,peak", [("100M:100.1M:100", -1, 0), ("100M:100.2M:1k", 0, 0),
                                           ("100M:100.1M:100", 9, 0), ("100M:100.1M:100", -1, 1),
                                           ("88M:108M:1k", -1, 1), ("100M:102.4M:19", -1, 1),
                                           ("box13", None, 0), ("box13", None, 1), ("fir14", None, 0)])
def test_guard_front_ends_and_peak_hold(scan_mod, port_oracle, freq, fir, peak):
    """narrow boxcar (ds = 28), -F 0, -F 9, and peak hold on the u8, decimated and large paths; decimated images on
    the large path (N >= 8192) behind a boxcar and a -F 9 chain"""
    from rtlsdr_b200.planner import plan_scan
    pd = dict(LARGE_DECIMATED[freq]) if freq in LARGE_DECIMATED else plan_scan(freq, 0.0, None if fir < 0 else
                                                                              fir).as_dict()
    pd["peak_hold"] = peak
    pd["tune_count"] = min(pd["tune_count"], 3)
    n = 1 << pd["bin_e"]
    w = port_oracle.window_coefs("hamming", n)
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=w, guard_bits=True)
    try:
        for rep in range(2):
            reads, hops = make_reads(port_oracle.lib, pd, 2, SYNTH_XORSHIFT, seed=11 + rep)
            want_avg, want_smp, _ = oracle_guard(port_oracle, pd, w, reads, hops)
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
            check_report(g.collect_all(), pd, want_avg, want_smp, (freq, fir, peak, rep))
    finally:
        g.close()


@pytest.mark.parametrize("bin_e", [10, 17])
def test_guard_async_report_and_short_reads(scan_mod, port_oracle, bin_e):
    """ASYNC_REPORT with collect_device (back-to-back intervals), and SHORT_READS"""
    import torch
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=2)
    w = port_oracle.window_coefs("hamming", n)
    g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=True, async_report=True)
    s = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=True, short_reads=True)
    try:
        for rep in range(3):
            reads, hops = make_reads(port_oracle.lib, plan, 2, SYNTH_BIASED, seed=rep, param=15)
            want_avg, want_smp, _ = oracle_guard(port_oracle, plan, w, reads, hops)
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
            out = [torch.zeros((2, n), dtype=torch.int64, device="cuda"),
                   torch.zeros(2, dtype=torch.int32, device="cuda"),
                   torch.zeros((2, g.db_count), dtype=torch.float64, device="cuda")]
            g.collect_device(*[o.data_ptr() for o in out])
            torch.cuda.synchronize()
            torch.cuda.ExternalStream(g.get_report_stream()).synchronize()
            check_report([o.cpu().numpy() for o in out], plan, want_avg, want_smp, ("async", rep))
        # a short read replaces the first bytes of the hop's previous read (what rtl_power's buffer holds)
        reads, hops = make_reads(port_oracle.lib, plan, 1, SYNTH_BIASED, seed=9, param=30)
        full = reads.copy()
        for r, h in zip(reads, hops):
            s.submit(int(h), r)
        short = full.copy()
        short[:, :plan["buf_len"] // 3] = 255 - short[:, :plan["buf_len"] // 3]
        for r, h in zip(short, hops):
            s.submit(int(h), r[:plan["buf_len"] // 3])
        want_avg, want_smp, _ = oracle_guard(port_oracle, plan, w, np.concatenate([full, short]),
                                             np.concatenate([hops, hops]))
        check_report(s.collect_all(), plan, want_avg, want_smp, "short")
    finally:
        g.close()
        s.close()


@pytest.mark.parametrize("bin_e", [5, 12, 13, 17])
def test_guard_sk(scan_mod, port_oracle, bin_e):
    """S2 equals the oracle's 128-bit sums and the SK rows equal the host sk_from_moments bit for bit"""
    from test_sk import sk_py
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=2, crop=0.2)
    w = port_oracle.window_coefs("rectangle", n)
    g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=True, spectral_kurtosis=True)
    try:
        for rep in range(2):
            reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e + rep, param=25)
            reads[1] = full_scale(plan["buf_len"])
            want_avg, want_smp, want_s2 = oracle_guard(port_oracle, plan, w, reads, hops)
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
            avg, smp, db, s2, sk = g.collect_sk()
            check_report((avg, smp, db), plan, want_avg, want_smp, ("sk", rep))
            assert np.array_equal(s2.reshape(want_s2.shape), want_s2)
            want_sk, _, _ = expected_sk_rows(want_avg, want_smp, want_s2, bin_e, 0.2, 1, f=sk_py)
            assert all(same_bits(a, b) for a, b in zip(sk.ravel(), want_sk.ravel()))
    finally:
        g.close()


@pytest.mark.parametrize("bin_e,sk", [(10, False), (10, True), (17, False), (17, True)])
def test_guard_merge_three_handles(scan_mod, port_oracle, bin_e, sk):
    """three handles merged with merge_device / merge_sk_device give the bytes of one handle"""
    import torch
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=2)
    w = port_oracle.window_coefs("blackman", n)
    kw = dict(window_coefs=w, guard_bits=True, spectral_kurtosis=sk)
    one = scan_mod.GpuScan.from_plan(plan, **kw)
    parts = [scan_mod.GpuScan.from_plan(plan, **kw) for _ in range(3)]
    try:
        reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=bin_e, param=40)
        for i, (r, h) in enumerate(zip(reads, hops)):
            one.submit(int(h), r)
            parts[i % 3].submit(int(h), r)
        words = 2 * n + 1 + (4 * n if sk else 0)
        sets = torch.zeros((2, words), dtype=torch.int64, device="cuda")
        for k, p in enumerate(parts[1:]):
            avg_p, smp_p = sets[k, :2 * n].data_ptr(), sets[k, 2 * n:].data_ptr()
            if sk:
                p.collect_sk_device(avg_p, smp_p, None, sets[k, 2 * n + 1:].data_ptr(), None)
            else:
                p.collect_device(avg_p, smp_p, None)
        torch.cuda.synchronize()
        stride = words * 8
        if sk:
            parts[0].merge_sk_device(sets[0, :2 * n].data_ptr(), sets[0, 2 * n:].data_ptr(),
                                     sets[0, 2 * n + 1:].data_ptr(), 2, stride)
            a, b = parts[0].collect_sk(), one.collect_sk()
        else:
            parts[0].merge_device(sets[0, :2 * n].data_ptr(), sets[0, 2 * n:].data_ptr(), 2, stride)
            a, b = parts[0].collect_all(), one.collect_all()
        assert all(np.ascontiguousarray(x).tobytes() == np.ascontiguousarray(y).tobytes() for x, y in zip(a, b))
        want_avg, want_smp, _ = oracle_guard(port_oracle, plan, w, reads, hops)
        assert np.array_equal(b[0], want_avg) and np.array_equal(b[1], want_smp)
    finally:
        for g in [one] + parts:
            g.close()


def test_guard_iir_and_level_stats(scan_mod, port_oracle):
    """-s iir on a guard handle: three reports against the smoothing of the oracle's scaled linear values; the soft-AGC
    byte counts equal those of a handle without the flag"""
    import math
    bin_e, alpha = 10, 0.25
    n = 1 << bin_e
    plan = plan_dict(bin_e, tune_count=2, crop=0.1)
    w = port_oracle.window_coefs("hamming", n)
    g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=True, iir_alpha=alpha, level_stats=True)
    q = scan_mod.GpuScan.from_plan(plan, window_coefs=w, level_stats=True)
    state = None
    try:
        for rep in range(3):
            reads, hops = make_reads(port_oracle.lib, plan, 3, SYNTH_BIASED, seed=20 + rep, param=10 + 20 * rep)
            reads[0, :40] = 255
            want_avg, want_smp, _ = oracle_guard(port_oracle, plan, w, reads, hops)
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
                q.submit(int(h), r)
            assert [g.level_stats(h) for h in range(2)] == [q.level_stats(h) for h in range(2)]
            avg, smp, db = g.collect_all()
            q.collect_all()
            assert np.array_equal(avg, want_avg) and np.array_equal(smp, want_smp)
            i1, i2 = plan_i(plan)
            d = np.array([[float(want_avg[h, 1 if ((i + n // 2) & (n - 1)) == 0 else (i + n // 2) & (n - 1)])
                           * 2.0 ** -8 / plan["rate"] / float(want_smp[h]) for i in range(i1, i2 + 1)]
                          for h in range(2)])
            state = d if state is None else state + alpha * (d - state)
            want = np.array([[10 * math.log10(v) for v in row] + [10 * math.log10(row[-1])] for row in state])
            assert db_close(db, want), rep
    finally:
        g.close()
        q.close()


def plan_i(plan):
    n = 1 << plan["bin_e"]
    return int(n * plan["crop"] * 0.5), (n - 1) - int(n * plan["crop"] * 0.5)


def test_guard_flag_leaves_other_handles_alone(scan_mod, port_oracle):
    """the same bytes on a handle without the flag give the Q15 results and CSV, beside a guard handle"""
    from scan_cases import expected
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan("88M:108M:1k", 0.2, None)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    n = 1 << pd["bin_e"]
    w = port_oracle.window_coefs("hamming", n)
    reads, hops = make_reads(port_oracle.lib, pd, 2, SYNTH_XORSHIFT, seed=2)
    plain, guard = (scan_mod.GpuScan.from_plan(pd, window_coefs=w, guard_bits=gb) for gb in (False, True))
    try:
        low, high, step = plan.csv_columns()
        for g in (plain, guard):
            g.set_csv_columns(low, high, step)
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
        text = plain.collect_csv("2026-01-01, 00:00:00, ")
        for r, h in zip(reads, hops):
            plain.submit(int(h), r)
        avg, smp, db = plain.collect_all()
        want = expected(port_oracle, pd, w, reads, hops)
        assert np.array_equal(avg, want[0]) and np.array_equal(smp, want[1]) and db_close(db, want[2])
        rows = "".join("2026-01-01, 00:00:00, " + plan.csv_row(h, int(want[1][h]), want[2][h])
                       for h in range(pd["tune_count"]))
        assert bytes(text).decode() == rows
        gtext = guard.collect_csv("2026-01-01, 00:00:00, ")
        ga, gs, _ = oracle_guard(port_oracle, pd, w, reads, hops)
        grows = "".join("2026-01-01, 00:00:00, " + plan.csv_row(h, int(gs[h]), want_report(pd, ga, gs)[h])
                        for h in range(pd["tune_count"]))
        assert bytes(gtext).decode() == grows
    finally:
        plain.close()
        guard.close()


# ---- sweep_main --guard-bits and rtl_power_gpu -G ------------------------------------------------------------

def _run_sweep_main(args, out, world, timeout=600):
    base = [sys.executable]
    if world > 1:
        base += ["-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                 "--master-port", str(29500 + os.getpid() % 2000), "-m", "rtlsdr_b200.sweep_main",
                 "--backend", "gloo", "--device", "0"]
    else:
        base += ["-m", "rtlsdr_b200.sweep_main"]
    r = subprocess.run(base + args + ["-o", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]
    return out.read_text()


@pytest.mark.parametrize("args,shard", [
    (["-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "--synth", "biased", "--seed", "4", "--param", "17"], "hops"),
    (["-f", "100M:102.4M:2400", "--synth", "biased", "--seed", "2", "--param", "33"], "reads"),
])
def test_sweep_main_guard_bits(scan_mod, tmp_path, args, shard):
    """power and SK files identical at 1, 2 and 3 gloo ranks on one GPU, and different from the Q15 rows"""
    args = args + ["--sweeps", "5", "--intervals", "2", "--shard", shard, "--guard-bits"]
    want = _run_sweep_main(args, tmp_path / "p1.csv", 1)
    sk1 = tmp_path / "sk1.csv"
    assert _run_sweep_main(args + ["--sk", str(sk1)], tmp_path / "p1sk.csv", 1) == want
    want_sk = sk1.read_text()
    assert len(want) > 100 and len(want_sk) > 100
    q15 = _run_sweep_main([a for a in args if a != "--guard-bits"], tmp_path / "q.csv", 1)
    assert q15 != want
    for world in (2, 3):
        skw = tmp_path / f"sk{world}.csv"
        assert _run_sweep_main(args + ["--sk", str(skw)], tmp_path / f"p{world}.csv", world) == want
        assert skw.read_text() == want_sk


def cli_want_rows(port_oracle, rng_, peak, sk):
    """the rows rtl_power_gpu -G -1 must print for RTLSDR_SYNTH_MODE=biased, seed 3, param 21, 4 sweeps: the guard
    oracle's bins, counts and S2, its dB rows and host-formatted SK rows"""
    from test_sk import sk_py
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(rng_, 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = peak
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    reads, hops = make_reads(port_oracle.lib, pd, 4, SYNTH_BIASED, seed=3, param=21)
    avg, smp, s2 = oracle_guard(port_oracle, pd, w, reads, hops)
    db = want_report(pd, avg, smp)
    rows = [CLI_STAMP + plan.csv_row(h, int(smp[h]), db[h]) for h in range(pd["tune_count"])]
    sk_rows = []
    if sk:
        vals, _, _ = expected_sk_rows(avg, smp, s2, pd["bin_e"], pd["crop"], pd["downsample"], f=sk_py)
        for h in range(pd["tune_count"]):
            prefix = rows[h].split(", ")[:6]
            sk_rows.append(", ".join(prefix + ["nan" if v != v else "%.4f" % v for v in vals[h]]) + "\n")
    return "".join(rows), "".join(sk_rows)


CLI_STAMP = "2026-01-01, 00:00:00, "


@pytest.mark.parametrize("rng_,peak,sk,extra", [("88M:108M:25k", 0, True, []), ("100M:102.4M:2400", 0, False, []),
                                                ("88M:108M:25k", 1, False, ["-P", "-R", "5"])])
def test_cli_guard_bits(scan_mod, port_oracle, tmp_path, rng_, peak, sk, extra):
    """rtl_power_gpu -G, with -t 1 and -t 3: power (and -K) rows byte-identical to the host-formatted guard oracle
    rows -- on a multi-hop plan, on a one-hop plan (more workers than hops: the reads are dealt and merged; -K needs
    every read of a hop on one worker, so that plan runs without it) and with -P -R"""
    from rtlsdr_b200 import _build
    _build.build_host()
    exe = os.path.join(_build.HOST_BUILD, "rtl_power_gpu")
    env = dict(os.environ, RTLSDR_SYNTH_MODE="biased", RTLSDR_SYNTH_SEED="3", RTLSDR_SYNTH_PARAM="21",
               RTL_POWER_PASSES="4", RTL_POWER_TIMESTAMP="2026-01-01, 00:00:00", RTLSDR_GPU_DEVICES="0,0,0")
    want, want_sk = cli_want_rows(port_oracle, rng_, peak, sk)
    assert len(want) > 100 and (not sk or len(want_sk) > 100)
    for t in ("1", "3"):
        out, skf = tmp_path / f"p{t}.csv", tmp_path / f"sk{t}.csv"
        cmd = [exe, "-f", rng_, "-c", "20%", "-w", "hamming", "-1", "-G", "-t", t] + extra
        cmd += ["-K", str(skf)] if sk else []
        r = subprocess.run(cmd + [str(out)], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        assert out.read_text() == want, t
        if sk:
            assert skf.read_text() == want_sk, t


# ---- what the guard bits buy ----------------------------------------------------------------------------------

def noise_reads(n_reads, buf_len, sigma, seed, tone=0.0, bin_frac=0.1):
    rng = np.random.default_rng(seed)
    k = np.arange(buf_len // 2)
    sig = tone * np.exp(2j * np.pi * bin_frac * k)
    out = np.empty((n_reads, buf_len), dtype=np.uint8)
    for r in range(n_reads):
        z = sig + rng.normal(0, sigma, buf_len // 2) + 1j * rng.normal(0, sigma, buf_len // 2)
        iq = np.empty(buf_len)
        iq[0::2], iq[1::2] = z.real, z.imag
        out[r] = np.clip(np.rint(iq + 127.0), 0, 255).astype(np.uint8)
    return out


@pytest.mark.parametrize("bin_e,n_reads", [(12, 64), (17, 16)])
def test_guard_noise_floor_and_sk(scan_mod, port_oracle, bin_e, n_reads):
    """u8 noise of sigma = 3 counts, rectangle window: the mean guard dB of the interior bins is within 0.3 dB of the
    float64 expectation 10 log10(2 * sigma^2 * 256^2 / N / rate * ds) (the Q15 value is printed, not asserted), and
    the mean guard SK is within 0.05 of 1"""
    n = 1 << bin_e
    plan = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=1, rate=2400000)
    w = port_oracle.window_coefs("rectangle", n)
    reads = noise_reads(n_reads, plan["buf_len"], 3.0, bin_e)
    res = {}
    for gb in (False, True):
        g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=gb, spectral_kurtosis=True)
        try:
            for r in reads:
                g.submit(0, r)
            avg, smp, db, s2, sk = g.collect_sk()
        finally:
            g.close()
        inner = slice(n // 8, n // 2 - n // 8)
        res[gb] = (float(np.mean(db[0][inner])), float(np.nanmean(sk[0][inner])))
    # E|X|^2 of fix_fft's X = DFT(x)/N with x = 256 (u - 127): 2 sigma^2 256^2 / N per block, in the scale csv_dbm
    # divides by rate and samples (ds = 1 per block)
    q = 2 * 3.0 ** 2 * 256.0 ** 2 / n
    expect_db = 10 * np.log10(q / plan["rate"])
    print(f"bin_e {bin_e}: float64 expectation {expect_db:.2f} dB, guard {res[True][0]:.2f} dB (SK {res[True][1]:.3f}),"
          f" Q15 {res[False][0]:.2f} dB (SK {res[False][1]:.3f})")
    assert abs(res[True][0] - expect_db) < 0.3
    assert abs(res[True][1] - 1.0) < 0.05


def test_guard_strong_tone_reads_the_same_db(scan_mod, port_oracle):
    bin_e, n = 12, 4096
    plan = plan_dict(bin_e, tune_count=1)
    w = port_oracle.window_coefs("rectangle", n)
    reads = noise_reads(8, 16384, 2.0, 5, tone=90.0, bin_frac=512 / 4096)
    peaks = []
    for gb in (False, True):
        g = scan_mod.GpuScan.from_plan(plan, window_coefs=w, guard_bits=gb)
        try:
            for r in reads:
                g.submit(0, r)
            _, _, db = g.collect_all()
        finally:
            g.close()
        peaks.append(float(db[0][:-1].max()))
    assert abs(peaks[0] - peaks[1]) < 0.05, peaks
