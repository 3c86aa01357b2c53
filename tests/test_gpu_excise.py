"""Spectral-kurtosis RFI excision on the GPU (RTLSDR_GPU_FLAG_SK_EXCISION): the clean sums, clean block counts and
folded samples equal the Python fold oracle fed with the exact per-sub-integration sums of a twin SK handle; the
excised dB and flag rows equal their host evaluation; an excision handle's ordinary reports are byte-identical to a
plain SK handle's; and the excision behaves on noise, bursts and steady tones."""
import math

import numpy as np
import pytest

from oracles import SYNTH_BIASED, SYNTH_XORSHIFT
from scan_cases import make_reads, plan_dict
from test_excise import State, ex, fold_oracle, report_oracle  # noqa: F401  (ex: fixture)
from test_sk import oracle_sk

pytestmark = pytest.mark.gpu
STAMP = "2026-01-01, 00:00:00, "
INF = float("inf")


@pytest.fixture(scope="module")
def scan_mod():
    import rtlsdr_b200.scan as s
    s.load_library()
    return s


def feed(handles, pd, reads, hops, how, scan_mod):
    """the reads (pass-major, every hop once per pass) into every handle through one submit route"""
    tc, b = pd["tune_count"], pd["buf_len"]
    if how == "submit":
        for g in handles:
            for r, h in zip(reads, hops):
                g.submit(int(h), r)
        return
    passes = len(reads) // tc
    if how == "reads":                                         # hop visits in a shuffled order
        order = np.random.default_rng(len(reads)).permutation(len(reads))
        reads, hops = reads[order], hops[order]
    if how in ("batch", "reads"):
        pinned = scan_mod.PinnedBuffer(reads.nbytes)
        pinned.array[:] = reads.reshape(-1)
        for g in handles:
            if how == "batch":
                g.submit_batch(0, tc, passes, pinned.ptr, tc * b, b)
            else:
                g.submit_reads(hops, pinned.ptr)
            g.sync()
        return
    import torch
    dev = torch.from_numpy(np.ascontiguousarray(reads)).cuda()
    torch.cuda.synchronize()
    for g in handles:
        g.submit_device(0, tc, passes, dev.data_ptr(), tc * b, b)
        g.sync()


def add_sums(st, avg, smp, s2):
    for h in range(st.hops):
        st.smp[h] += int(smp[h])
        for j in range(st.n):
            st.S1[h][j] += int(avg[h, j])
            st.S2[h][j] += int(s2[h, j, 0]) | (int(s2[h, j, 1]) << 64)


def check_excised(ex, g, st, pd, guard, n_db):
    c1, b1, smp, db, fl = g.excised_report()
    assert np.array_equal(c1, np.array(st.c1, dtype=np.int64))
    assert np.array_equal(b1, np.array(st.b1, dtype=np.int64))
    assert np.array_equal(smp, np.array(st.snap_smp))
    i1, i2 = db_range(pd)
    wdb, wfl = report_oracle(st, pd["bin_e"], i1, i2, pd["rate"], pd["downsample"], guard)
    assert db.shape[1] == n_db
    assert np.array_equal(np.isnan(db), np.isnan(wdb)) and not np.signbit(db[np.isnan(db)]).any()
    ok = ~np.isnan(wdb)
    assert np.array_equal(db[ok] == -INF, wdb[ok] == -INF)
    fin = ok & np.isfinite(wdb)
    assert np.allclose(db[fin], wdb[fin], rtol=1e-12, atol=1e-12)
    assert fl.tobytes() == wfl.tobytes()                      # one correctly rounded division
    return db, fl


def db_range(pd):
    """csv_dbm's printed bins [i1, i2] (rtl_power.c:741-748), as the library's scan_shape computes them"""
    n = 1 << pd["bin_e"]
    crop = pd["crop"]
    i1 = int(float(n) * crop * 0.5)
    i2 = (n - 1) - int(float(n) * crop * 0.5)
    return i1, i2


CASES = [  # (label, plan, window, route, guard)
    ("u8-5", plan_dict(5, tune_count=3), "rectangle", "submit", False),
    ("u8-10-guard", plan_dict(10, tune_count=2, crop=0.2), "hamming", "batch", True),
    ("u8-12", plan_dict(12, tune_count=2), "hamming", "reads", False),
    ("large-13-guard", plan_dict(13, buf_len=2 << 13, tune_count=2), "hamming", "device", True),
    ("large-17", plan_dict(17, buf_len=2 << 17, tune_count=1, crop=0.1), "hamming", "batch", False),
    ("boxcar-ds28", "100M:100.1M:100", "hamming", "device", False),
    ("fir9-guard", "100M:100.3M:3k", "hamming", "submit", True),
]


def case_plan(spec):
    if isinstance(spec, dict):
        return dict(spec)
    from rtlsdr_b200.planner import plan_scan
    fir = 9 if spec == "100M:100.3M:3k" else None
    pd = plan_scan(spec, 0.0 if fir is None else 0.1, fir).as_dict()
    pd["peak_hold"] = 0
    return pd


@pytest.mark.parametrize("label,spec,window,how,guard", CASES, ids=[c[0] for c in CASES])
def test_excision_matches_oracle(scan_mod, ex, port_oracle, label, spec, window, how, guard):
    """two intervals: one fold, then three uneven folds and a chunk after the last fold (ordinary rows only)"""
    pd = case_plan(spec)
    n = 1 << pd["bin_e"]
    w = port_oracle.window_coefs(window, n)
    e = scan_mod.GpuScan.from_plan(pd, window_coefs=w, sk_excision=True, guard_bits=guard)
    t = scan_mod.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True, guard_bits=guard)
    st = State(pd["tune_count"], n)
    flagged = clean = 0
    try:
        for interval, chunks in enumerate(([4], [1, 3, 2, 1])):
            for c, passes in enumerate(chunks):
                reads, hops = make_reads(port_oracle.lib, pd, passes, SYNTH_XORSHIFT if c % 2 else SYNTH_BIASED,
                                         seed=17 * interval + c, param=20 + c)
                if c == 1:
                    reads[0, 0::64] = 255                      # a burst in one read
                feed((e, t), pd, reads, hops, how, scan_mod)
                avg, smp, _, s2, _ = t.collect_sk()            # the sub-integration's exact sums
                if not guard and c == 0 and pd["downsample"] == 1:
                    want = oracle_sk(port_oracle, pd, w, reads, hops)
                    assert np.array_equal(avg, want[0]) and np.array_equal(s2, want[2])
                add_sums(st, avg, smp, s2)
                if interval == 1 and c == len(chunks) - 1:
                    break                                      # submitted after the last fold
                e.excise_fold(1.0, 1.5)
                fold_oracle(ex, st, 1.0, 1.5, pd["downsample"])
            _, fl = check_excised(ex, e, st, pd, guard, e.db_count)
            flagged += int(np.nansum(fl > 0))
            clean += int(np.nansum(fl < 1))
            total = np.array(st.S1, dtype=np.int64)
            avg, smp, _, _, _ = e.collect_sk()                 # the ordinary report still has every read
            assert np.array_equal(avg, total) and np.array_equal(smp, np.array(st.smp))
            st.zero()
            c1, b1, fsmp, _, _ = e.excised_report()            # the read-and-zero cleared the excision state
            assert not c1.any() and not b1.any() and not fsmp.any()
        assert flagged and clean
    finally:
        e.close()
        t.close()


def test_excision_handle_reports_are_unchanged(scan_mod, port_oracle):
    """the same reads into an excision handle (folded in between) and a plain SK handle: collect_sk, collect_csv
    and collect_sk_csv print the same bytes"""
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan("88M:108M:25k", 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    e = scan_mod.GpuScan.from_plan(pd, window_coefs=w, sk_excision=True)
    t = scan_mod.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True)
    try:
        for g in (e, t):
            g.set_csv_columns(*plan.csv_columns())
        for what in ("sk", "csv", "sk_csv"):
            for c in range(3):
                reads, hops = make_reads(port_oracle.lib, pd, 1, SYNTH_BIASED, seed=len(what) + c, param=30)
                feed((e, t), pd, reads, hops, "submit", scan_mod)
                e.excise_fold()
            if what == "sk":
                a, b = e.collect_sk(), t.collect_sk()
                assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
            elif what == "csv":
                assert e.collect_csv(STAMP) == t.collect_csv(STAMP)
            else:
                assert e.collect_sk_csv(STAMP) == t.collect_sk_csv(STAMP)
    finally:
        e.close()
        t.close()


def test_excised_device_report_and_text(scan_mod, port_oracle):
    """excised_report_device() writes what excised_report() returns; excised_csv() prints those values like the
    host printf, with the folded samples as the count column; a peek zeroes nothing"""
    import torch
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan("88M:108M:25k", 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=w, sk_excision=True)
    try:
        g.set_csv_columns(*plan.csv_columns())
        for c in range(3):
            reads, hops = make_reads(port_oracle.lib, pd, 2, SYNTH_BIASED, seed=c, param=25)
            feed((g,), pd, reads, hops, "submit", scan_mod)
            g.excise_fold(1.0, 1.0)
        tc, dbc = pd["tune_count"], g.db_count
        _, _, smp, db, fl = g.excised_report()
        d_db = torch.zeros((tc, dbc), dtype=torch.float64, device="cuda")
        d_fl = torch.zeros((tc, dbc), dtype=torch.float64, device="cuda")
        d_smp = torch.zeros(tc, dtype=torch.int32, device="cuda")
        g.excised_report_device(d_db.data_ptr(), d_fl.data_ptr(), d_smp.data_ptr())
        g.sync()
        assert d_db.cpu().numpy().tobytes() == db.tobytes()
        assert d_fl.cpu().numpy().tobytes() == fl.tobytes()
        assert np.array_equal(d_smp.cpu().numpy(), smp)
        text, ftext = g.excised_csv(STAMP)
        rows = "".join(STAMP + plan.csv_row(h, int(smp[h]), db[h]) for h in range(tc))
        assert text.decode() == rows
        frows = []
        for h in range(tc):
            prefix = (STAMP + plan.csv_row(h, int(smp[h]), db[h])).split(", ")[:6]
            frows.append(", ".join(prefix + ["nan" if v != v else "%.4f" % v for v in fl[h]]) + "\n")
        assert ftext.decode() == "".join(frows)
        assert g.excised_csv(STAMP, flags=False) == (text, None)
        assert g.excised_report()[3].tobytes() == db.tobytes()
    finally:
        g.close()


def test_excision_refusals(scan_mod):
    import torch
    g = scan_mod.GpuScan(2, 10, 16384, sk_excision=True)
    sk = scan_mod.GpuScan(2, 10, 16384, spectral_kurtosis=True)
    try:
        d_avg = torch.zeros((2, 1024), dtype=torch.int64, device="cuda")
        d_smp = torch.zeros(2, dtype=torch.int32, device="cuda")
        d_s2 = torch.zeros((2, 1024, 2), dtype=torch.int64, device="cuda")
        d_db_ptr = d_avg.data_ptr()
        for call in (lambda: g.merge_device(d_avg.data_ptr(), d_smp.data_ptr()),
                     lambda: g.merge_sk_device(d_avg.data_ptr(), d_smp.data_ptr(), d_s2.data_ptr()),
                     lambda: g.excise_fold(float("nan"), 3.0), lambda: g.excise_fold(3.0, -1.0),
                     lambda: sk.excise_fold(), lambda: sk.excised_report(), lambda: sk.excised_csv(STAMP),
                     lambda: sk.excised_report_device(d_db_ptr)):
            with pytest.raises(scan_mod.ScanError) as e:
                call()
            assert e.value.code == -2
        with pytest.raises(scan_mod.ScanError) as e:
            g.excised_report_device(d_avg.data_ptr() + 4)
        assert e.value.code == -8
        with pytest.raises(scan_mod.ScanError) as e:
            g.excised_csv(STAMP)                               # no column table
        assert e.value.code == -2
        g.excise_fold(INF, INF)
        g.excise_fold(0.0, 0.0)
    finally:
        g.close()
        sk.close()


# ---- statistics -------------------------------------------------------------------------------------------

def tone_reads(rng, n_reads, n, k0, amp, on, buf_len=16384):
    """uniform noise bytes plus, in the reads where on[i], a complex tone exactly on bin k0 of an n-point block"""
    t = np.arange(buf_len // 2)
    reads = rng.integers(127 - 60, 128 + 60, (n_reads, buf_len)).astype(np.float64)
    for i in range(n_reads):
        if on[i]:
            ph = 2 * np.pi * k0 * t / n + rng.uniform(0, 2 * np.pi)
            reads[i, 0::2] += amp * np.cos(ph)
            reads[i, 1::2] += amp * np.sin(ph)
    return np.clip(np.round(reads), 0, 255).astype(np.uint8)


def test_burst_is_excised(scan_mod):
    """u8 noise, a strong tone in 2 of 16 sub-integrations (M = 256): the tone bin is flagged exactly 2/16, its
    excised dB is the noise level, while its ordinary dB is far above"""
    bin_e, k0 = 5, 5
    n = 1 << bin_e
    col = (k0 + n // 2) % n
    rng = np.random.default_rng(11)
    g = scan_mod.GpuScan(1, bin_e, 16384, sk_excision=True)
    try:
        on = [i in (3, 11) for i in range(16)]
        for r in tone_reads(rng, 16, n, k0, 50.0, on):
            g.submit(0, r)
            g.excise_fold(3.0, 3.0)
        _, _, _, xdb, fl = g.excised_report()
        _, _, db, _, _ = g.collect_sk()
        noise = np.delete(np.arange(n + 1), [col, n // 2, n])    # neither the tone, the DC bin nor the duplicate
        expect = float(np.median(db[0, noise]))
        print(f"tone bin: flagged {fl[0, col]:.4f}, excised {xdb[0, col]:.2f} dB, ordinary {db[0, col]:.2f} dB, "
              f"noise {expect:.2f} dB, noise bins flagged {np.mean(fl[0, noise]):.4f}")
        assert fl[0, col] == 0.125
        assert abs(xdb[0, col] - expect) < 0.5
        assert db[0, col] > expect + 5                         # 2 of 16 sub-integrations at about +15 dB
    finally:
        g.close()


@pytest.mark.parametrize("bin_e,guard,reads_per_fold,folds", [(6, False, 1, 32), (10, False, 8, 8),
                                                             (12, True, 32, 8), (17, True, 64, 4)])
def test_noise_flag_rate(scan_mod, bin_e, guard, reads_per_fold, folds):
    """uniform u8 noise, symmetric 3 sigma at M >= 64: the mean flag fraction stays below 2 %"""
    n = 1 << bin_e
    buf_len = 16384 if bin_e <= 12 else 2 * n
    rng = np.random.default_rng(bin_e)
    g = scan_mod.GpuScan(1, bin_e, buf_len, sk_excision=True, guard_bits=guard)
    try:
        import torch
        reads = torch.from_numpy(rng.integers(0, 256, (folds * reads_per_fold, buf_len), dtype=np.uint8)).cuda()
        for f in range(folds):
            g.submit_device(0, 1, reads_per_fold, reads[f * reads_per_fold].data_ptr(), buf_len, buf_len)
            g.excise_fold(3.0, 3.0)
        _, b1, smp, _, fl = g.excised_report()
        M = int(smp[0]) // folds
        assert M >= 64
        rate = float(np.nanmean(fl[0]))
        print(f"bin_e {bin_e} guard {guard}: M = {M}, mean flag fraction of noise {rate:.4%}")
        assert rate < 0.02
    finally:
        g.close()


def test_steady_tone(scan_mod):
    """a steady tone is flagged in every sub-integration with k_low = 3 and in none with k_low = +inf, where the
    excised dB equals the ordinary dB"""
    bin_e, k0 = 5, 7
    n = 1 << bin_e
    col = (k0 + n // 2) % n
    rng = np.random.default_rng(3)
    reads = tone_reads(rng, 8, n, k0, 50.0, [True] * 8)
    for k_low, want in ((3.0, 1.0), (INF, 0.0)):
        g = scan_mod.GpuScan(1, bin_e, 16384, sk_excision=True)
        try:
            for r in reads:
                g.submit(0, r)
                g.excise_fold(k_low, 3.0)
            _, _, _, xdb, fl = g.excised_report()
            _, _, db, _, _ = g.collect_sk()
            assert fl[0, col] == want
            if want == 0.0:
                assert math.isclose(xdb[0, col], db[0, col], rel_tol=1e-6)
            else:
                assert math.isnan(xdb[0, col])
        finally:
            g.close()


# ---- rtl_power_gpu ----------------------------------------------------------------------------------------

def test_cli_excise_files(scan_mod, port_oracle, tmp_path):
    """rtl_power_gpu -X/-Y -M 2: the excised and flag rows of a handle folded every 2 sweeps, the same with one and
    two workers; the power file does not change with -X; the refusals"""
    import os
    import subprocess
    from rtlsdr_b200 import _build
    from rtlsdr_b200.planner import plan_scan
    _build.build_host()
    exe = os.path.join(_build.HOST_BUILD, "rtl_power_gpu")
    env = dict(os.environ, RTLSDR_SYNTH_MODE="biased", RTLSDR_SYNTH_SEED="3", RTLSDR_SYNTH_PARAM="21",
               RTL_POWER_PASSES="5", RTL_POWER_TIMESTAMP="2026-01-01, 00:00:00", RTLSDR_GPU_DEVICES="0,0")
    args = ["-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "-1"]
    files = {}
    for t, extra in ((1, []), (1, ["-X", "x", "-Y", "y", "-M", "2", "-k", "1:2"]),
                     (2, ["-X", "x", "-Y", "y", "-M", "2", "-k", "1:2"])):
        d = tmp_path / f"t{t}{len(extra)}"
        d.mkdir()
        r = subprocess.run([exe] + args + ["-t", str(t)] + extra + ["out"], env=env, cwd=d, capture_output=True,
                           text=True, timeout=120)
        assert r.returncode == 0, r.stderr
        files[(t, bool(extra))] = {f: (d / f).read_bytes() for f in os.listdir(d)}
    assert files[(1, True)]["out"] == files[(1, False)]["out"]
    assert files[(1, True)] == files[(2, True)]
    plan = plan_scan("88M:108M:25k", 0.2)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    reads, hops = make_reads(port_oracle.lib, pd, 5, SYNTH_BIASED, seed=3, param=21)
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=w, sk_excision=True)
    try:
        g.set_csv_columns(*plan.csv_columns())
        for p in range(5):
            for r, h in zip(reads[p * pd["tune_count"]:(p + 1) * pd["tune_count"]], hops):
                g.submit(int(h), r)
            if p % 2 == 1 or p == 4:
                g.excise_fold(1.0, 2.0)
        x, y = g.excised_csv(STAMP)
    finally:
        g.close()
    assert files[(1, True)]["x"] == x and files[(1, True)]["y"] == y
    for bad in (["-X", "x", "-P"], ["-Y", "y"], ["-X", "x", "-k", "-1"]):
        r = subprocess.run([exe] + args + bad + [str(tmp_path / "o")], env=env, capture_output=True, text=True,
                           timeout=120)
        assert r.returncode == 1, bad
    for bad in (["-f", "100M:100.1M:100", "-t", "2"],         # more workers than hops (read-sharded merge)
                ["-f", "100M:104M:1M"]):                      # 1-bin (rms) hops
        r = subprocess.run([exe] + bad + ["-X", str(tmp_path / "x"), str(tmp_path / "o")], env=env,
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 1 and "-X" in r.stderr, bad
        assert not (tmp_path / "x").exists()


# ---- sweep_main --excise ----------------------------------------------------------------------------------

SWEEP_ARGS = ["-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "--synth", "biased", "--seed", "4", "--param", "17",
              "--sweeps", "5", "--intervals", "2"]


def one_handle_excised_rows(scan_mod, sweeps, intervals, chunk, k_low, k_high):
    """excised_csv() of one handle fed the synthetic source's reads, folded after every `chunk` sweeps (None: the
    fewest sweeps giving 64 FFT blocks, from the library's geometry)"""
    from rtlsdr_b200.planner import host_library, plan_scan, synth_cube
    plan = plan_scan("88M:108M:25k", host_library().rp_atofp(b"20%"), None)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    tc, b = pd["tune_count"], pd["buf_len"]
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=scan_mod.window_coefs("hamming", 1 << pd["bin_e"]),
                                   sk_excision=True)
    cube = scan_mod.PinnedBuffer(sweeps * tc * b)
    x, y = [], []
    try:
        if chunk is None:
            chunk = g.excise_sweeps()
            assert chunk == -(-64 // g.blocks_per_read)
        g.set_csv_columns(*plan.csv_columns())
        for j in range(intervals):
            synth_cube(cube.ptr, 3, 4, 17, tc, 0, tc, j * sweeps, sweeps, b)
            for p0 in range(0, sweeps, chunk):
                g.submit_batch(0, tc, min(chunk, sweeps - p0), cube.ptr + p0 * tc * b, tc * b, b)
                g.excise_fold(k_low, k_high)
            xt, yt = g.excised_csv(STAMP)
            x.append(xt.decode())
            y.append(yt.decode())
            g.collect_sk()
    finally:
        g.close()
        cube.free()
    return "".join(x), "".join(y)


def test_sweep_main_excise(scan_mod, tmp_path):
    """--excise/--excise-flags at 1-3 gloo ranks (and with --random-hops) write the rows of one handle folded every K
    sweeps; the power and SK files are the same with and without --excise"""
    from test_gpu_sk_multi import _run_sweep_main
    sk0 = tmp_path / "sk0.csv"
    plain = _run_sweep_main(SWEEP_ARGS + ["--sk", str(sk0)], tmp_path / "plain.csv", 1)
    want_x, want_y = one_handle_excised_rows(scan_mod, 5, 2, 2, 1.0, 2.0)
    assert len(want_x) > 100 and len(want_y) > 100
    for world, extra in ((1, []), (2, []), (3, []), (2, ["--random-hops", "5"])):
        d = tmp_path / f"w{world}{len(extra)}"
        d.mkdir()
        args = SWEEP_ARGS + extra + ["--sk", str(d / "sk.csv"), "--excise", str(d / "x.csv"), "--excise-flags",
                                     str(d / "y.csv"), "--excise-sweeps", "2", "--excise-sigma", "1:2"]
        power = _run_sweep_main(args, d / "p.csv", world)
        assert power == plain, (world, extra)
        assert (d / "sk.csv").read_text() == sk0.read_text()
        assert (d / "x.csv").read_text() == want_x, (world, extra)
        assert (d / "y.csv").read_text() == want_y, (world, extra)
    # the default K: the fewest sweeps giving every hop 64 FFT blocks per sub-integration
    d = tmp_path / "default"
    d.mkdir()
    _run_sweep_main(SWEEP_ARGS + ["--excise", str(d / "x.csv")], d / "p.csv", 1)
    assert (d / "x.csv").read_text() == one_handle_excised_rows(scan_mod, 5, 2, None, 3.0, 3.0)[0]


def test_sweep_main_excise_refusals(scan_mod, tmp_path):
    import os
    import subprocess
    import sys
    from test_gpu_sk_multi import ROOT
    for extra, what in ((["-f", "100M:102.4M:300", "--shard", "reads"], "--shard reads"),
                        (["-f", "100M:102.4M:300", "-P"], "-P"), (["-f", "100M:104M:1M"], "rms"),
                        (["-f", "88M:108M:25k", "--excise-sigma", "-1"], "--excise-sigma")):
        r = subprocess.run([sys.executable, "-m", "rtlsdr_b200.sweep_main"] + extra + ["--excise", str(tmp_path / "x")],
                           cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert r.returncode != 0 and "--excise" in r.stderr and what in r.stderr, (extra, r.stderr[-500:])
        assert not (tmp_path / "x").exists()
    r = subprocess.run([sys.executable, "-m", "rtlsdr_b200.sweep_main", "-f", "88M:108M:25k", "--excise-flags",
                        str(tmp_path / "y")], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--excise-flags needs --excise" in r.stderr
    assert not os.path.exists(tmp_path / "y")
