#!/usr/bin/env python
"""A/B timing of kernel variants: RTLSDR_GPU_SCAN_LIB=<other build> python tools/ab_small.py [config ...]
Device-resident steps, CUDA events on the handle's stream, >= 50 ms per measurement (same method as bench.py)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import rtlsdr_b200.scan as rs  # noqa: E402
from rtlsdr_b200.planner import plan_scan  # noqa: E402

CONFIGS = {
    "cfg5": ("24M:1457.6M:700", 0.0, "rectangle", None, 0, 256),
    "cfg5s": ("24M:1457.6M:700", 0.0, "rectangle", None, 0, 32),     # one GPU's share at N = 8
    "cfg5n8": ("24M:203.2M:700", 0.0, "rectangle", None, 0, 256),     # exactly one GPU's share at N = 8: 64 hops x 256 sweeps
    "cfg5n4": ("24M:382.4M:700", 0.0, "rectangle", None, 0, 256),     # one GPU's share at N = 4
    "cfg2": ("88M:108M:1k", 0.2, "hamming", None, 0, 377),
    "cfg3": ("24M:1766M:1k", 0.0, "rectangle", 9, 0, 64),
    "cfg1": ("100M:102.4M:2400", 0.0, "rectangle", None, 0, 293),
    "cfg4": ("100M:102.4M:19", 0.0, "blackman-harris", None, 1, 256),
    "box28": ("100M:100.1M:100", 0.0, "rectangle", None, 0, 8192),
    "box14pk": ("100M:100.2M:50", 0.0, "rectangle", None, 1, 4096),  # 4096 bins, ds = 14, peak hold: stream kernel <12,1,2,2>
    "f9": ("100M:100.1M:100", 0.0, "blackman", 9, 0, 8192),
    "rms": ("100M:110M:1M", 0.0, "rectangle", None, 0, 4096),
    "rms1k": ("100M:110M:1M", 0.0, "rectangle", None, 0, 1024),
    "rms16k": ("100M:110M:1M", 0.0, "rectangle", None, 0, 16384),
    "box28x4": ("100M:100.1M:100", 0.0, "rectangle", None, 0, 32768),
}


def run(name):
    base, _, override = name.partition(":")          # "cfg5:32" = config 5 with 32 sweeps per step
    freq, crop, window, fir, peak, passes = CONFIGS[base]
    if override:
        passes = int(override)
    pd = plan_scan(freq, crop, fir).as_dict()
    pd["peak_hold"] = peak
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    g = rs.GpuScan.from_plan(pd, window_coefs=rs.window_coefs(window, n) if pd["bin_e"] else None)
    stream = torch.cuda.ExternalStream(g.get_stream())
    step_bytes = passes * tc * b
    n_sets = max(1, -(-(300 << 20) // step_bytes))
    dev_in = torch.randint(0, 256, (n_sets, passes, tc, b), dtype=torch.uint8, device="cuda")
    out = torch.zeros(tc * (n + g.db_count + 1), dtype=torch.int64, device="cuda")
    p_avg = out.data_ptr()
    p_db = p_avg + tc * n * 8
    p_smp = p_db + tc * g.db_count * 8

    def step(i):
        g.submit_device(0, tc, passes, dev_in[i % n_sets].data_ptr(), tc * b, b)
        g.collect_device(p_avg, p_smp, p_db)

    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    best, total, done = 1e9, 0.0, 0
    while total < 60.0:
        k = max(1, int(10 / max(best, 0.01))) if done else 3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(k):
            step(done + i)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = min(best, ms / k)
        total += ms
        done += k
    g.close()
    print(f"{name:6s} {os.path.basename(rs.lib_path()):32s} best {best:9.4f} ms/step  {step_bytes / 2 / (best * 1e-3) / 1e6:12.0f} Msamples/s  "
          f"mean {total / done:9.4f} ms  {step_bytes / 2 / (total / done * 1e-3) / 1e6:12.0f} Msamples/s", flush=True)


if __name__ == "__main__":
    for name in (sys.argv[1:] or ["cfg5", "cfg2"]):
        run(name)
