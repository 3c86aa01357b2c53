"""What the guard-bit transform (RTLSDR_GPU_FLAG_GUARD_BITS) costs against the Q15 transform.

    python tools/guard_rate.py [--rounds 5] [--out profiles/r07_guard_rate.json]

For each workload two handles of the same configuration, guard bits off and on, are fed the same device-resident
random bytes (rotating sets of >= 300 MB, larger than L2) with submit_device(); rounds alternate off / on, each
round >= 60 ms of back-to-back steps timed with CUDA events on the handle's stream.  Only the transform is timed
(no report in the window).  Workloads:
  cfg5    config 5, 512 hops x 4096 bins, 256 sweeps per step (u8 small path)
  cfg4    config 4's shape without -P, 2^17 bins (large path)
  cfg4p   config 4's shape with -P (peak hold)
  box28   narrow boxcar ds = 28 at 1024 bins (guard handles take the staged boxcar route)
  f9      -F 9, ds = 16 at 1024 bins
Records the GPU name and power limit beside the numbers.  Needs a CUDA device: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg5": ("24M:1457.6M:700", 0.0, "rectangle", None, 256),
    "cfg4": ("100M:102.4M:19", 0.0, "blackman-harris", None, 256),
    "cfg4p": ("100M:102.4M:19", 0.0, "blackman-harris", None, 256),
    "box28": ("100M:100.1M:100", 0.0, "rectangle", None, 8192),
    "f9": ("100M:100.1M:100", 0.0, "blackman", 9, 8192),
}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi failed: {e}"


def run(torch, rs, name, rounds):
    from rtlsdr_b200.planner import plan_scan
    freq, crop, window, fir, passes = WORKLOADS[name]
    pd = plan_scan(freq, crop, fir).as_dict()
    pd["peak_hold"] = 1 if name == "cfg4p" else 0
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    w = rs.window_coefs(window, n)
    handles = {gb: rs.GpuScan.from_plan(pd, window_coefs=w, guard_bits=gb) for gb in (False, True)}
    step_bytes = passes * tc * b
    n_sets = max(1, -(-(300 << 20) // step_bytes))
    dev_in = torch.randint(0, 256, (n_sets, passes, tc, b), dtype=torch.uint8, device="cuda")
    res = {sk: [] for sk in handles}
    done = {sk: 0 for sk in handles}

    def window_ms(sk, min_ms):
        g = handles[sk]
        stream = torch.cuda.ExternalStream(g.get_stream())
        total, k_done, k = 0.0, 0, 2
        while total < min_ms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(k):
                g.submit_device(0, tc, passes, dev_in[done[sk] % n_sets].data_ptr(), tc * b, b)
                done[sk] += 1
            e1.record(stream)
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
            k_done += k
            k = max(1, int(20 / max(total / k_done, 0.01)))
        return total / k_done

    for sk in handles:                                # warm-up of every kernel and table
        window_ms(sk, 20.0)
    for _ in range(rounds):
        for sk in (False, True):
            res[sk].append(window_ms(sk, 60.0))
    for g in handles.values():
        g.close()
    rate = lambda ms: step_bytes / 2 / (ms * 1e-3) / 1e9  # noqa: E731  G samples/s (complex)
    out = {"workload": name, "range": freq, "fir": fir, "bin_e": pd["bin_e"], "downsample": pd["downsample"],
           "hops": tc, "sweeps_per_step": passes}
    for sk, key in ((False, "guard_off"), (True, "guard_on")):
        ms = res[sk]
        out[key] = {"ms_per_step": [round(m, 4) for m in ms], "best_gsps": round(rate(min(ms)), 2),
                    "mean_gsps": round(rate(sum(ms) / len(ms)), 2)}
    out["on_over_off_best"] = round(min(res[False]) / min(res[True]), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("workloads", nargs="*", default=list(WORKLOADS))
    a = ap.parse_args()
    import torch
    import rtlsdr_b200.scan as rs
    if not torch.cuda.is_available():
        sys.exit("guard_rate.py needs a CUDA device")
    rs.load_library()
    doc = {"gpu": gpu_info(), "method": "submit_device steps, CUDA events, >= 60 ms per round, guard bits off / on alternated",
           "results": [run(torch, rs, w, a.rounds) for w in a.workloads]}
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
