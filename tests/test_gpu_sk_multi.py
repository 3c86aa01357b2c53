"""Spectral kurtosis across handles and GPUs: collect_sk_device against collect_sk, merge_sk_device of three handles
against one handle and the oracle, the SK rows' text formatted on the GPU (format_sk_csv_device, collect_sk_csv),
sweep_main --sk in both shard modes at 1-3 gloo ranks on one GPU, and rtl_power_gpu -K -t 2."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracles import SYNTH_BIASED
from scan_cases import make_reads, plan_dict
from test_sk import full_scale, oracle_sk
from test_sk_text import sk_row_text

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAMP = "2026-01-01, 00:00:00, "


@pytest.fixture(scope="module")
def scan_mod():
    import rtlsdr_b200.scan as s
    s.load_library()
    return s


def sk_handles(scan_mod, pd, w, count):
    return [scan_mod.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True) for _ in range(count)]


def submit_all(g, reads, hops):
    for r, h in zip(reads, hops):
        g.submit(int(h), r)


@pytest.mark.parametrize("bin_e", [4, 10, 12, 13, 17])
def test_collect_sk_device_equals_collect_sk(scan_mod, port_oracle, bin_e):
    """twin SK handles, three reports (read-and-zero), the second with full-scale reads (at 16 bins, rectangle
    window, 512 blocks per read: S2 high words non-zero; fix_fft's scaling keeps larger transforms below 2^64);
    the third report passes NULL for some outputs"""
    import torch
    n = 1 << bin_e
    pd = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=3, crop=0.2)
    w = port_oracle.window_coefs("rectangle" if bin_e == 4 else "hamming", n)
    a, b = sk_handles(scan_mod, pd, w, 2)
    tc, dbc = pd["tune_count"], a.db_count
    try:
        for rep in range(3):
            reads, hops = make_reads(port_oracle.lib, pd, 2, SYNTH_BIASED, seed=7 * bin_e + rep, param=23)
            if rep == 1:
                reads[:3] = full_scale(pd["buf_len"])
            submit_all(a, reads, hops)
            submit_all(b, reads, hops)
            want = a.collect_sk()
            out = [torch.full((tc, n), -1, dtype=torch.int64, device="cuda"),
                   torch.full((tc,), -1, dtype=torch.int32, device="cuda"),
                   torch.full((tc, dbc), -1.0, dtype=torch.float64, device="cuda"),
                   torch.full((tc, n, 2), 7, dtype=torch.int64, device="cuda"),
                   torch.full((tc, dbc), -1.0, dtype=torch.float64, device="cuda")]
            keep = [True] * 5 if rep < 2 else [False, True, False, True, True]
            b.collect_sk_device(*[o.data_ptr() if k else None for o, k in zip(out, keep)])
            torch.cuda.synchronize()
            for o, wnt, k in zip(out, want, keep):
                if k:
                    assert o.cpu().numpy().tobytes() == np.ascontiguousarray(wnt).tobytes()
            if rep == 1 and bin_e == 4:
                assert want[3][..., 1].any()
        # both handles are zero again
        empty_a, empty_b = a.collect_sk(), b.collect_sk()
        assert not empty_b[0].any() and not empty_b[1].any() and not empty_b[3].any()
        assert all(x.tobytes() == y.tobytes() for x, y in zip(empty_a, empty_b))
    finally:
        a.close()
        b.close()


def set_layout(tc, n):
    """one external set: S1 int64 [tc * n], counts int32 [tc] padded to 8 bytes, S2 u64 [tc * n][2] -- in words"""
    smp_at = tc * n
    s2_at = smp_at + (tc + 1) // 2
    return smp_at, s2_at, s2_at + 2 * tc * n


@pytest.mark.parametrize("bin_e,tc", [(4, 2), (10, 1), (12, 3), (14, 2)])
@pytest.mark.parametrize("where", ["device", "pinned"])
def test_merge_sk_device_three_handles_equal_one(scan_mod, port_oracle, bin_e, tc, where):
    """each of three handles takes a third of the reads; merge_sk_device folds handles 1 and 2 into handle 0:
    S1, counts, dB, S2 and SK equal one handle that saw every read, and the oracle's sums"""
    import torch
    n = 1 << bin_e
    pd = plan_dict(bin_e, buf_len=16384 if bin_e <= 12 else 2 * n, tune_count=tc, crop=0.1)
    w = port_oracle.window_coefs("rectangle" if bin_e == 4 else "blackman-harris", n)
    reads, hops = make_reads(port_oracle.lib, pd, 6, SYNTH_BIASED, seed=bin_e + tc, param=19)
    reads[tc: 3 * tc] = full_scale(pd["buf_len"])          # passes 1 and 2: two handles' S2 reach the high word
    hs = sk_handles(scan_mod, pd, w, 4)
    one, parts = hs[0], hs[1:]
    smp_at, s2_at, words = set_layout(tc, n)
    pinned = None
    try:
        submit_all(one, reads, hops)
        third = (np.arange(len(reads)) // tc) % 3          # handle i gets passes i, i + 3
        for i, g in enumerate(parts):
            submit_all(g, reads[third == i], hops[third == i])
        if where == "device":
            sets = torch.zeros((2, words), dtype=torch.int64, device="cuda")
            base = sets.data_ptr()
            for s, g in enumerate(parts[1:]):
                p = base + s * words * 8
                g.collect_sk_device(p, p + smp_at * 8, None, p + s2_at * 8, None)
                g.sync()
        else:
            pinned = scan_mod.PinnedBuffer(2 * words * 8)
            base = pinned.ptr
            for s, g in enumerate(parts[1:]):
                o = s * words * 8
                avg = pinned.view(np.int64, (tc, n), o)
                smp = pinned.view(np.int32, (tc,), o + smp_at * 8)
                s2 = pinned.view(np.uint64, (tc, n, 2), o + s2_at * 8)
                g._check(g.lib.rtlsdr_gpu_scan_collect_sk(g.h, avg.ctypes.data, smp.ctypes.data, None,
                                                          s2.ctypes.data, None), "collect_sk")
        parts[0].merge_sk_device(base, base + smp_at * 8, base + s2_at * 8, 2, words * 8)
        got, want = parts[0].collect_sk(), one.collect_sk()
        for x, y in zip(got, want):
            assert x.tobytes() == y.tobytes()
        o_avg, o_smp, o_s2 = oracle_sk(port_oracle, pd, w, reads, hops)
        assert np.array_equal(got[0], o_avg) and np.array_equal(got[1], o_smp) and np.array_equal(got[3], o_s2)
        if bin_e == 4:
            assert got[3][..., 1].any()
    finally:
        for g in hs:
            g.close()
        if pinned is not None:
            pinned.free()


def test_merge_sk_device_argument_checks(scan_mod):
    import torch
    g = scan_mod.GpuScan(2, 10, 16384, spectral_kurtosis=True)
    plain = scan_mod.GpuScan(2, 10, 16384)
    L = g.lib
    buf = torch.zeros(8192, dtype=torch.int64, device="cuda")
    p = buf.data_ptr()
    try:
        assert L.rtlsdr_gpu_scan_merge_sk_device(g.h, p, p, None, 1, 0) == -1
        assert L.rtlsdr_gpu_scan_merge_sk_device(g.h, p, p, p, 0, 0) == -2
        assert L.rtlsdr_gpu_scan_merge_sk_device(g.h, p, p, p, 2, 0) == -2
        assert L.rtlsdr_gpu_scan_merge_sk_device(g.h, p, p, p + 4, 1, 0) == -8
        assert L.rtlsdr_gpu_scan_merge_sk_device(g.h, p, p, p, 2, 12) == -8
        assert L.rtlsdr_gpu_scan_merge_sk_device(plain.h, p, p, p, 1, 0) == -2
        assert L.rtlsdr_gpu_scan_collect_sk_device(plain.h, p, p, p, p, p) == -2
        assert L.rtlsdr_gpu_scan_sk_csv_capacity(plain.h, 1, 10) == -2
    finally:
        g.close()
        plain.close()


def expected_rows(plan, smp, db, sk, hop0=0):
    """the power rows and SK rows rtl_power_gpu -K writes, built like test_gpu_sk.py::test_cli_sk_file"""
    rows, sk_rows = [], []
    low, high, step = plan.csv_columns()
    for h in range(len(smp)):
        rows.append(STAMP + plan.csv_row(hop0 + h, int(smp[h]), db[h]))
        sk_rows.append(sk_row_text(STAMP, low[hop0 + h], high[hop0 + h], step, int(smp[h]), sk[h]))
    return "".join(rows), "".join(sk_rows)


@pytest.mark.parametrize("freq,crop", [("88M:108M:25k", 0.2), ("100M:102.4M:300", 0.0)])
def test_sk_text_on_the_gpu(scan_mod, port_oracle, freq, crop):
    """collect_sk_csv and format_sk_csv_device print the expected rows; the power text equals collect_csv's"""
    import torch
    from rtlsdr_b200.planner import plan_scan
    plan = plan_scan(freq, crop)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    w = port_oracle.window_coefs("hamming", 1 << pd["bin_e"])
    a, b, c = sk_handles(scan_mod, pd, w, 3)
    plain = scan_mod.GpuScan.from_plan(pd, window_coefs=w)
    tc, n = pd["tune_count"], 1 << pd["bin_e"]
    try:
        for g in (b, c, plain):
            g.set_csv_columns(*plan.csv_columns())
        for rep in range(2):
            reads, hops = make_reads(port_oracle.lib, pd, 3, SYNTH_BIASED, seed=rep, param=30)
            if rep == 1:
                reads[:] = 127                           # S1 = 0: every SK value NaN
            for g in (a, b, c, plain):
                submit_all(g, reads, hops)
            _, smp, db, _, sk = a.collect_sk()
            want, want_sk = expected_rows(plan, smp, db, sk)
            text, sk_text = b.collect_sk_csv(STAMP)
            assert text.decode() == want and sk_text.decode() == want_sk
            assert plain.collect_csv(STAMP) == text
            # the device formatter over a collect_sk_device() report, from row 1 on
            d_smp = torch.zeros(tc, dtype=torch.int32, device="cuda")
            d_sk = torch.zeros((tc, c.db_count), dtype=torch.float64, device="cuda")
            c.collect_sk_device(None, d_smp.data_ptr(), None, None, d_sk.data_ptr())
            r0 = 1 if tc > 1 else 0
            rows = tc - r0
            cap = c.sk_csv_capacity(rows, len(STAMP))
            lens_at = (cap + 7) // 8 * 8
            out = torch.zeros(lens_at + 8, dtype=torch.uint8, device="cuda")
            lens = out[lens_at:].view(torch.int64)
            c.format_sk_csv_device(STAMP, r0, rows, d_sk[r0:].data_ptr(), c.db_count, d_smp[r0:].data_ptr(),
                                   out.data_ptr(), cap, lens.data_ptr())
            torch.cuda.synchronize()
            m = int(lens.item())
            assert out[:m].cpu().numpy().tobytes().decode() == expected_rows(plan, smp[r0:], db[r0:], sk[r0:], r0)[1]
        # errors: capacity, no column table, handle without the flag
        small = np.empty(b.sk_csv_capacity(tc, len(STAMP)) - 1, dtype=np.uint8)
        with pytest.raises(scan_mod.ScanError) as e:
            b.collect_sk_csv(STAMP, sk_out=small)
        assert e.value.code == -4
        with pytest.raises(scan_mod.ScanError) as e:
            a.collect_sk_csv(STAMP)
        assert e.value.code == -2
        with pytest.raises(scan_mod.ScanError) as e:
            c.format_sk_csv_device(STAMP, 0, tc, d_sk.data_ptr(), c.db_count, d_smp.data_ptr(), out.data_ptr(), 16,
                                   lens.data_ptr())
        assert e.value.code == -4
        with pytest.raises(scan_mod.ScanError) as e:
            plain.collect_sk_csv(STAMP, sk_out=np.empty(1 << 20, dtype=np.uint8))
        assert e.value.code == -2
        with pytest.raises(scan_mod.ScanError) as e:
            plain.format_sk_csv_device(STAMP, 0, tc, d_sk.data_ptr(), c.db_count, d_smp.data_ptr(), out.data_ptr(),
                                       cap, lens.data_ptr())
        assert e.value.code == -2
    finally:
        for g in (a, b, c, plain):
            g.close()


# ---- sweep_main --sk and rtl_power_gpu -K -t 2 ----------------------------------------------------------------

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


def one_handle_sk_rows(scan_mod, args, sweeps, intervals):
    """the SK rows of one handle fed the synthetic source's reads for every (sweep, hop), via collect_sk"""
    from rtlsdr_b200.planner import host_library, plan_scan, synth_cube
    rng_ = args[args.index("-f") + 1]
    synth = args[args.index("--synth") + 1] if "--synth" in args else "xorshift"
    seed = int(args[args.index("--seed") + 1]) if "--seed" in args else 0
    param = int(args[args.index("--param") + 1]) if "--param" in args else 0
    window = args[args.index("-w") + 1] if "-w" in args else "rectangle"
    crop = host_library().rp_atofp((args[args.index("-c") + 1] if "-c" in args else "0").encode())
    plan = plan_scan(rng_, crop, None)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    tc, b = pd["tune_count"], pd["buf_len"]
    mode = ["xorshift", "counter", "const", "biased", "tone"].index(synth)
    g = scan_mod.GpuScan.from_plan(pd, window_coefs=scan_mod.window_coefs(window, 1 << pd["bin_e"]),
                                   spectral_kurtosis=True)
    cube = scan_mod.PinnedBuffer(sweeps * tc * b)
    low, high, step = plan.csv_columns()
    rows = []
    try:
        for j in range(intervals):
            synth_cube(cube.ptr, mode, seed, param, tc, 0, tc, j * sweeps, sweeps, b)
            g.submit_batch(0, tc, sweeps, cube.ptr, tc * b, b)
            g.sync()
            _, smp, _, _, sk = g.collect_sk()
            rows += [sk_row_text("2026-01-01, 00:00:00, ", low[h], high[h], step, int(smp[h]), sk[h]) for h in range(tc)]
    finally:
        g.close()
        cube.free()
    return "".join(rows)


@pytest.mark.parametrize("args,shard,worlds", [
    (["-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "--synth", "biased", "--seed", "4", "--param", "17"],
     "hops", (2, 3)),
    (["-f", "100M:102.4M:2400", "--synth", "biased", "--seed", "2", "--param", "33"], "reads", (2, 3)),
    (["-f", "100M:102.4M:300", "-w", "blackman-harris", "--seed", "6"], "reads", (2,)),
])
def test_sweep_main_sk(scan_mod, tmp_path, args, shard, worlds):
    """SK files identical across world sizes and equal to one handle's collect_sk rows; power CSV unchanged"""
    sweeps, intervals = 5, 3
    args = args + ["--sweeps", str(sweeps), "--intervals", str(intervals), "--shard", shard]
    plain = _run_sweep_main(args, tmp_path / "plain.csv", 1)
    want_sk = one_handle_sk_rows(scan_mod, args, sweeps, intervals)
    assert len(want_sk) > 100
    for world in (1,) + worlds:
        sk_path = tmp_path / f"sk{world}.csv"
        power = _run_sweep_main(args + ["--sk", str(sk_path)], tmp_path / f"p{world}.csv", world)
        assert power == plain
        assert sk_path.read_text() == want_sk


def test_sweep_main_sk_refusals(scan_mod, tmp_path):
    for extra, what in ((["-f", "100M:102.4M:300", "-P"], "-P"), (["-f", "100M:104M:1M"], "rms")):
        r = subprocess.run([sys.executable, "-m", "rtlsdr_b200.sweep_main"] + extra + ["--sk", str(tmp_path / "x")],
                           cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert r.returncode != 0 and "--sk" in r.stderr and what in r.stderr
        assert not (tmp_path / "x").exists()


def test_cli_sk_two_workers(scan_mod, tmp_path):
    """rtl_power_gpu -K -t 2 on a multi-hop plan: both files identical to -t 1"""
    from rtlsdr_b200 import _build
    _build.build_host()
    exe = os.path.join(_build.HOST_BUILD, "rtl_power_gpu")
    env = dict(os.environ, RTLSDR_SYNTH_MODE="biased", RTLSDR_SYNTH_SEED="3", RTLSDR_SYNTH_PARAM="21",
               RTL_POWER_PASSES="4", RTL_POWER_REPORTS="3", RTL_POWER_TIMESTAMP="2026-01-01, 00:00:00",
               RTLSDR_GPU_DEVICES="0,0")
    got = []
    for t in ("1", "2"):
        out, skf = tmp_path / f"p{t}.csv", tmp_path / f"sk{t}.csv"
        r = subprocess.run([exe, "-f", "88M:108M:25k", "-c", "20%", "-w", "hamming", "-t", t, "-K", str(skf),
                            str(out)], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        got.append((out.read_text(), skf.read_text()))
    assert len(got[0][0]) > 1000 and len(got[0][1]) > 1000 and got[0] == got[1]
