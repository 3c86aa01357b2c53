"""What rtl_power's CSV text costs per integration interval, host printf versus the GPU formatter.

    python tools/csv_rate.py [--reps 5] [--sweep-main] [--baseline-tree DIR] > profiles/csv_rate.json

For BASELINE configs 3 (-f 24M:1766M:1k -F 9, 623 hops x 4096 bins) and 5 (-f 24M:1457.6M:700, 512 hops x 4096
bins) on one GPU, two handles are fed the same reads and timed from the collect to the rows in host memory:
  host  collect_all() (epilogue + dB doubles to the host) then stamp + rp_csv_row() per hop: how sweep_main
        and rtl_power_gpu printed the rows before the GPU formatter
  gpu   collect_csv(): epilogue + csv_rows_kernel + csv_pack_kernel, text to the host
Both produce the same bytes (checked).  `kernel_us` is the formatter alone (csv_rows_kernel + csv_pack_kernel via
format_csv_device on a collect_device report), CUDA events over repeated launches on the handle's stream.
`transform_beside_format` times the transform kernels of one handle with and without a second handle formatting
on its own stream at the same time (the alternative to formatting behind the exchange on the handle's stream).
--sweep-main times `sweep_main -f 24M:1766M:1k --sweeps 64 --intervals 8` end to end (and the same command from
--baseline-tree, e.g. a checkout of the parent commit with its library built).
--sk measures the spectral-kurtosis rows instead, on two spectral_kurtosis=True handles fed the same reads:
  host  collect_sk() then the power rows through rp_csv_row() and the SK rows through Python's "%.4f" (the bytes
        rtl_power_gpu -K printed with host printf before collect_sk_csv; Python's formatter stands in for printf)
  gpu   collect_sk_csv(): both texts formatted on the GPU, only text to the host
and with --sweep-main times the sweep_main command above with and without `--sk FILE`, alternated.
Records the GPU name and power limit beside the numbers.  Needs a CUDA device: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAMP = "2026-01-01, 00:00:00, "
CONFIGS = {3: ("24M:1766M:1k", 0.0, 9, 64), 5: ("24M:1457.6M:700", 0.0, None, 256)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi failed: {e}"


def feed(torch, pd, handles, sweeps, cube):
    tc, b = pd["tune_count"], pd["buf_len"]
    for g in handles:
        g.submit_device(0, tc, sweeps, cube.data_ptr(), tc * b, b)


def run_config(torch, rs, cfg, reps):
    from rtlsdr_b200.planner import plan_scan, synth_cube
    rng_, crop, fir, sweeps = CONFIGS[cfg]
    plan = plan_scan(rng_, crop, fir)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    w = rs.window_coefs("hamming", n)
    host_g = rs.GpuScan.from_plan(pd, window_coefs=w)
    gpu_g = rs.GpuScan.from_plan(pd, window_coefs=w)
    gpu_g.set_csv_columns(*plan.csv_columns())
    # one interval's reads from the synthetic source (xorshift), resident on the device
    pin = rs.PinnedBuffer(sweeps * tc * b)
    synth_cube(pin.ptr, 0, 1, 0, tc, 0, tc, 0, sweeps, b)
    cube = torch.from_numpy(pin.array).cuda()
    out = np.empty(gpu_g.csv_capacity(tc, len(STAMP)), dtype=np.uint8)
    host_ms, gpu_ms, same = [], [], True
    for _ in range(reps + 1):                       # the first round warms up both paths
        feed(torch, pd, (host_g, gpu_g), sweeps, cube)
        host_g.sync()
        gpu_g.sync()
        t0 = time.perf_counter()
        _, smp, db = host_g.collect_all()
        text_h = "".join(STAMP + plan.csv_row(h, int(smp[h]), db[h]) for h in range(tc)).encode()
        t1 = time.perf_counter()
        text_g = gpu_g.collect_csv(STAMP, out=out)
        t2 = time.perf_counter()
        same &= text_h == text_g
        host_ms.append((t1 - t0) * 1e3)
        gpu_ms.append((t2 - t1) * 1e3)
    host_ms, gpu_ms = host_ms[1:], gpu_ms[1:]

    # the formatter alone: format_csv_device on a collect_device report, CUDA events on the handle's stream
    feed(torch, pd, (gpu_g,), sweeps, cube)
    db_d = torch.empty(tc, gpu_g.db_count, dtype=torch.float64, device="cuda")
    smp_d = torch.empty(tc, dtype=torch.int32, device="cuda")
    gpu_g.collect_device(None, smp_d.data_ptr(), db_d.data_ptr())
    cap = gpu_g.csv_capacity(tc, len(STAMP))
    text_d = torch.empty(cap, dtype=torch.uint8, device="cuda")
    len_d = torch.empty(1, dtype=torch.int64, device="cuda")
    stream = torch.cuda.ExternalStream(gpu_g.get_stream())

    def fmt():
        gpu_g.format_csv_device(STAMP, 0, tc, db_d.data_ptr(), gpu_g.db_count, smp_d.data_ptr(), text_d.data_ptr(),
                                cap, len_d.data_ptr())
    fmt()
    gpu_g.sync()
    launches = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(launches):
        fmt()
    e1.record(stream)
    e1.synchronize()
    kernel_us = e0.elapsed_time(e1) * 1e3 / launches
    same &= text_d[: int(len_d.item())].cpu().numpy().tobytes() == text_g

    # the transform of one handle alone, and with another handle formatting on its own stream beside it
    def transform_ms(beside):
        host_g.set_timing(1)
        host_g.kernel_time()
        feed(torch, pd, (host_g,), sweeps, cube)
        if beside:
            for _ in range(launches):
                fmt()
        host_g.sync()
        gpu_g.sync()
        ms, k = host_g.kernel_time()
        host_g.collect_all(want_db=False)
        return ms
    transform_ms(False)
    alone = [transform_ms(False) for _ in range(reps)]
    beside = [transform_ms(True) for _ in range(reps)]
    host_g.set_timing(0)

    values = tc * gpu_g.db_count
    res = dict(config=cfg, range=rng_, hops=tc, bins=n, sweeps=sweeps, db_values=values, text_bytes=len(text_g),
               identical_bytes=bool(same), host_ms=[round(x, 2) for x in host_ms],
               gpu_ms=[round(x, 3) for x in gpu_ms], host_ms_median=round(float(np.median(host_ms)), 2),
               gpu_ms_median=round(float(np.median(gpu_ms)), 3),
               speedup=round(float(np.median(host_ms) / np.median(gpu_ms)), 1),
               host_ns_per_value=round(float(np.median(host_ms)) * 1e6 / values, 1),
               kernel_us=round(kernel_us, 1),
               transform_beside_format=dict(alone_ms=[round(x, 3) for x in alone],
                                            beside_ms=[round(x, 3) for x in beside]))
    for g in (host_g, gpu_g):
        g.close()
    pin.free()
    return res


def run_sk_config(torch, rs, cfg, reps):
    import math
    from rtlsdr_b200.planner import plan_scan, synth_cube
    rng_, crop, fir, sweeps = CONFIGS[cfg]
    plan = plan_scan(rng_, crop, fir)
    pd = plan.as_dict()
    pd["peak_hold"] = 0
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    w = rs.window_coefs("hamming", n)
    host_g = rs.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True)
    gpu_g = rs.GpuScan.from_plan(pd, window_coefs=w, spectral_kurtosis=True)
    gpu_g.set_csv_columns(*plan.csv_columns())
    low, high, step = plan.csv_columns()
    pin = rs.PinnedBuffer(sweeps * tc * b)
    synth_cube(pin.ptr, 0, 1, 0, tc, 0, tc, 0, sweeps, b)
    cube = torch.from_numpy(pin.array).cuda()
    out = np.empty(gpu_g.csv_capacity(tc, len(STAMP)), dtype=np.uint8)
    sk_out = np.empty(gpu_g.sk_csv_capacity(tc, len(STAMP)), dtype=np.uint8)
    host_ms, gpu_ms, same = [], [], True
    for _ in range(reps + 1):                       # the first round warms up both paths
        feed(torch, pd, (host_g, gpu_g), sweeps, cube)
        host_g.sync()
        gpu_g.sync()
        t0 = time.perf_counter()
        _, smp, db, _, sk = host_g.collect_sk()
        text_h = "".join(STAMP + plan.csv_row(h, int(smp[h]), db[h]) for h in range(tc)).encode()
        sk_h = "".join("%s%i, %i, %.2f, %i, " % (STAMP, low[h], high[h], step, smp[h])
                       + ", ".join("nan" if math.isnan(v) else "%.4f" % v for v in sk[h].tolist()) + "\n"
                       for h in range(tc)).encode()
        t1 = time.perf_counter()
        text_g, sk_g = gpu_g.collect_sk_csv(STAMP, out=out, sk_out=sk_out)
        t2 = time.perf_counter()
        same &= text_h == text_g and sk_h == sk_g
        host_ms.append((t1 - t0) * 1e3)
        gpu_ms.append((t2 - t1) * 1e3)
    host_ms, gpu_ms = host_ms[1:], gpu_ms[1:]
    values = tc * gpu_g.db_count
    res = dict(config=cfg, range=rng_, hops=tc, bins=n, sweeps=sweeps, values_per_text=values,
               text_bytes=len(text_g), sk_text_bytes=len(sk_g), identical_bytes=bool(same),
               host_ms=[round(x, 2) for x in host_ms], gpu_ms=[round(x, 3) for x in gpu_ms],
               host_ms_median=round(float(np.median(host_ms)), 2), gpu_ms_median=round(float(np.median(gpu_ms)), 3),
               speedup=round(float(np.median(host_ms) / np.median(gpu_ms)), 1))
    for g in (host_g, gpu_g):
        g.close()
    pin.free()
    return res


def time_sweep_main(tree, reps, extra=()):
    out, env = [], dict(os.environ, PYTHONPATH=tree, PYTHONDONTWRITEBYTECODE="1")
    cmd = [sys.executable, "-m", "rtlsdr_b200.sweep_main", "-f", "24M:1766M:1k", "--sweeps", "64",
           "--intervals", "8", "-o", os.devnull] + list(extra)
    for _ in range(reps):
        t0 = time.perf_counter()
        subprocess.run(cmd, cwd=tree, env=env, check=True, capture_output=True)
        out.append(round(time.perf_counter() - t0, 3))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweep-main", action="store_true")
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--sk", action="store_true", help="the spectral-kurtosis rows (see above)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("csv_rate: no CUDA device")
    import rtlsdr_b200.scan as rs
    rs.load_library()
    if args.sk:
        import tempfile
        res = dict(gpu=gpu_info(), sk_configs=[run_sk_config(torch, rs, c, args.reps) for c in (3, 5)])
        if args.sweep_main:
            sm = dict(without_sk_s=[], with_sk_s=[])
            with tempfile.TemporaryDirectory() as tmp:
                for _ in range(3):
                    sm["without_sk_s"] += time_sweep_main(ROOT, 1)
                    sm["with_sk_s"] += time_sweep_main(ROOT, 1, ["--sk", os.path.join(tmp, "sk.csv")])
            res["sweep_main_24M_1766M_1k_64x8"] = sm
        print(json.dumps(res, indent=1))
        return
    res = dict(gpu=gpu_info(), configs=[run_config(torch, rs, c, args.reps) for c in (3, 5)])
    if args.sweep_main:
        # alternate the two trees so that drift on a shared host hits both alike
        sm = dict(after_s=[], before_s=[])
        for _ in range(3):
            sm["after_s"] += time_sweep_main(ROOT, 1)
            if args.baseline_tree:
                sm["before_s"] += time_sweep_main(os.path.abspath(args.baseline_tree), 1)
        res["sweep_main_24M_1766M_1k_64x8"] = sm
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
