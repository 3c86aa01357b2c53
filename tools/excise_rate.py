"""What spectral-kurtosis excision (RTLSDR_GPU_FLAG_SK_EXCISION) costs.

    python tools/excise_rate.py [--rounds 5] [--out profiles/r08_excise_rate.json]

fold: one excise_fold_kernel at config 5's shape (512 hops x 4096 bins) and at 2^17 bins x 1 hop, each closing a
      sub-integration of M = 64 FFT blocks per hop (random reads submitted before every fold, outside the timed
      window), timed alone with CUDA events around the fold, L2 overwritten (a 512 MB memset) between the transform
      and the fold; the run records how many bins the timed folds flagged.  GB/s from the 96 bytes per
      bin the fold has to move (S1, S2, snapS1, snapS2, C1, B1 read; snapS1, snapS2, C1, B1 written) over the median
      time, against MEASURED_PEAKS.json's HBM bandwidth when the file exists (else the data sheet's 7.7 TB/s, so
      named).
interval: config 5, 256 sweeps per step from device-resident random bytes (rotating sets >= 300 MB) through
      submit_device(); an SK handle with one submit per step against an excision handle that submits K sweeps at a
      time with a fold after each chunk (K = 32 and 8); rounds alternate, >= 60 ms each, CUDA events on the
      handle's stream.  No report in the window.
Records the GPU name and power limit beside the numbers.  Needs a CUDA device: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BYTES_PER_BIN = 96
CFG5 = "24M:1457.6M:700"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi failed: {e}"


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            doc = json.load(f)
        for k, v in doc.items():
            if "hbm" in k.lower() or "bandwidth" in k.lower():
                return float(v if not isinstance(v, dict) else next(iter(v.values()))), f"MEASURED_PEAKS.json {k}"
    except Exception:  # noqa: BLE001
        pass
    return 7700.0, "data sheet (not measured)"


def fold_rate(torch, rs, tc, bin_e, buf_len, plan=None, iters=50, min_blocks=64):
    n = 1 << bin_e
    if plan is not None:
        g = rs.GpuScan.from_plan(plan, sk_excision=True)
    else:
        g = rs.GpuScan(tc, bin_e, buf_len, sk_excision=True)
    passes = g.excise_sweeps(min_blocks)
    dev_in = torch.randint(0, 256, (2, passes, tc, buf_len), dtype=torch.uint8, device="cuda")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.ExternalStream(g.get_stream())
    times = []
    for i in range(iters + 3):
        g.submit_device(0, tc, passes, dev_in[i & 1].data_ptr(), tc * buf_len, buf_len)   # M = passes * blocks
        with torch.cuda.stream(stream):
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        g.excise_fold(3.0, 3.0)
        e1.record(stream)
        torch.cuda.synchronize()
        if i >= 3:
            times.append(e0.elapsed_time(e1))
    _, b1, smp, _, _ = g.excised_report()
    g.close()
    folds = iters + 3
    M = int(smp[0]) // folds // (plan["downsample"] if plan else 1)
    flagged = 1.0 - float(b1.astype(np.int64).sum()) / (M * folds * b1.size)
    times.sort()
    ms = times[len(times) // 2]
    moved = BYTES_PER_BIN * tc * n
    return {"hops": tc, "bins": n, "blocks_per_fold": M, "flagged_share": round(flagged, 5),
            "bytes_per_fold": moved, "median_us": round(ms * 1e3, 2),
            "min_us": round(times[0] * 1e3, 2), "gbps": round(moved / (ms * 1e-3) / 1e9, 1)}


def interval_rate(torch, rs, rounds, chunks):
    from rtlsdr_b200.planner import plan_scan
    pd = plan_scan(CFG5, 0.0).as_dict()
    pd["peak_hold"] = 0
    tc, b, passes = pd["tune_count"], pd["buf_len"], 256
    handles = {0: rs.GpuScan.from_plan(pd, spectral_kurtosis=True)}
    for k in chunks:
        handles[k] = rs.GpuScan.from_plan(pd, sk_excision=True)
    step_bytes = passes * tc * b
    n_sets = max(1, -(-(300 << 20) // step_bytes))
    dev_in = torch.randint(0, 256, (n_sets, passes, tc, b), dtype=torch.uint8, device="cuda")
    done = {k: 0 for k in handles}
    res = {k: [] for k in handles}

    def step(k):
        g, base = handles[k], dev_in[done[k] % n_sets]
        done[k] += 1
        if k == 0:
            g.submit_device(0, tc, passes, base.data_ptr(), tc * b, b)
            return
        for p in range(0, passes, k):
            g.submit_device(0, tc, k, base[p].data_ptr(), tc * b, b)
            g.excise_fold(3.0, 3.0)

    def window_ms(k, min_ms):
        stream = torch.cuda.ExternalStream(handles[k].get_stream())
        total, n_done, m = 0.0, 0, 2
        while total < min_ms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(m):
                step(k)
            e1.record(stream)
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
            n_done += m
            m = max(1, int(20 / max(total / n_done, 0.01)))
        return total / n_done

    for k in handles:
        window_ms(k, 20.0)
    for _ in range(rounds):
        for k in handles:
            res[k].append(window_ms(k, 60.0))
    for g in handles.values():
        g.close()
    rate = lambda ms: step_bytes / 2 / (ms * 1e-3) / 1e9  # noqa: E731  G samples/s (complex)
    out = {"range": CFG5, "hops": tc, "bin_e": pd["bin_e"], "sweeps_per_step": passes,
           "sk_only": {"ms_per_step": [round(m, 4) for m in res[0]], "best_gsps": round(rate(min(res[0])), 2)}}
    for k in chunks:
        out[f"fold_every_{k}"] = {"ms_per_step": [round(m, 4) for m in res[k]], "best_gsps": round(rate(min(res[k])), 2),
                                  "overhead_best": round(min(res[k]) / min(res[0]) - 1, 4)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import rtlsdr_b200.scan as rs
    if not torch.cuda.is_available():
        sys.exit("excise_rate.py needs a CUDA device")
    rs.load_library()
    from rtlsdr_b200.planner import plan_scan
    pd = plan_scan(CFG5, 0.0).as_dict()
    pd["peak_hold"] = 0
    peak, peak_src = hbm_peak()
    folds = [fold_rate(torch, rs, pd["tune_count"], pd["bin_e"], pd["buf_len"], plan=pd),
             fold_rate(torch, rs, 1, 17, 2 << 17)]
    for f in folds:
        f["share_of_hbm_peak"] = round(f["gbps"] / peak, 4)
    doc = {"gpu": gpu_info(), "hbm_peak_gbps": peak, "hbm_peak_source": peak_src,
           "method": "fold: a sub-integration of M >= 64 FFT blocks submitted, a 512 MB memset, then events around one "
                     "fold, median of 50; interval: submit_device steps "
                     "of 256 sweeps, CUDA events, >= 60 ms per round, handles alternated",
           "fold": folds, "interval": interval_rate(torch, rs, a.rounds, (32, 8))}
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
