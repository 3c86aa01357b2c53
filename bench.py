#!/usr/bin/env python
"""bench.py -- throughput of rtl_power's per-hop scan pipeline on B200.

Metric (BASELINE.json): input Msamples/s (1 sample = 1 complex IQ pair = 2 input
bytes), whole job over all GPUs, plus the fraction of the HBM roofline.

Headline workload = BASELINE.json configs[4], the run SURVEY.md 8(d)(5) calls "the
roofline run": `-f 24M:1457.6M:700` = 512 hop streams x 4096 bins (rectangle),
256 sweeps per integration interval (2 GiB of uint8 IQ per step), hops SHARDED over
the N GPUs (512/256/128/64 per GPU at N = 1/2/4/8: strong scaling, no data-path
collective).  One "step" = one whole integration interval: every read of the
interval through the transform, the report epilogue (DC nuke, half swap, crop, dB)
on every rank, and ONE exchange of the spectra to rank 0 (rtlsdr_b200/sweep.py).
Input bytes are the synthetic source's xorshift stream, a pure function of
(hop, sweep) (host/synth_source.c), so the result does not depend on N:

  verify: outside the timed region the gathered int64 bins are FNV-hashed on rank 0 and
          compared (a) for sweep 0 alone with the reference-generated known-answer hash of
          SURVEY.md 8(c) and (b) for the whole interval with a 1-rank run of the same bytes.
  value : inputs already resident in HBM, CUDA-event timed on the launching stream,
          max over ranks, over exactly --steps steps.
  --dump-outputs DIR: the report of the last timed step (what a caller of the timed path
          receives) as DIR/avg.npy, db.npy, samples.npy in float64 (about 32 MiB in all).
  e2e   : the same interval through the public C ABI with HOST buffers:
          rtlsdr_gpu_scan_submit_batch() from pinned memory (H2D inside the timed
          region), the exchange, and the gathered report copied to host memory on rank 0.
  companions: BASELINE configs[2] (623 hops, sharded the same way, every N) and, at N = 1,
          configs[1] (round 1's headline) and the decimating / rms / large-FFT regimes.
  --impl reference : the reference's own CPU code (oracle/_ref, the unmodified
          rtl_power.c object) on all host cores, bounded sample per step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the bench leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# BASELINE configs[4]: the headline
RANGE, CROP, WINDOW, FIR = "24M:1457.6M:700", 0.0, "rectangle", None
SWEEPS = 256                 # sweeps per integration interval (SURVEY.md 8d: P >= 256)
WORKLOAD = "throughput_stress_512_hop_streams_4096bins_256_sweeps (BASELINE configs[4])"
KAT_P1 = 0x7b1c7343a9686225  # SURVEY.md 8(c): reference rtl_power, this range, 1 sweep, xorshift source
# BASELINE configs[2]: second sharded workload
RANGE3, FIR3, SWEEPS3, KAT3_P1 = "24M:1766M:1k", 9, 64, 0x074f712a23c886d1
# BASELINE configs[1]: round 1's headline, kept as an N = 1 companion
RANGE2, CROP2, WINDOW2, SWEEPS2 = "88M:108M:1k", 0.2, "hamming", 377
MIN_TIMED_MS = 50.0
SYNTH_XORSHIFT = 0


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def read_ncu():
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "10",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- reference arm

_REF = {}


def _ref_init(seed_base, rng, crop, window):
    """pool initializer: one configured reference instance per worker process"""
    import multiprocessing as mp
    from oracles import RefOracle, PortOracle, SYNTH_XORSHIFT as XS  # noqa
    ident = mp.current_process()._identity
    seed = seed_base + (ident[0] if ident else 0)
    try:
        r = RefOracle()
        r.configure(rng, crop, window)
        r.source(XS, seed, 0)
        r.scan(1)
        _REF.update(kind="reference", ref=r, per_pass=r.plan["tune_count"] * (r.plan["buf_len"] // 2))
    except Exception:
        # compiled reference missing: time the C restatement instead
        import numpy as np
        from rtlsdr_b200.planner import plan_scan
        p = PortOracle()
        plan = plan_scan(rng, crop).as_dict()
        plan["peak_hold"] = 0
        w = p.window_coefs(window, 1 << plan["bin_e"])
        rs = np.random.default_rng(seed)
        reads = rs.integers(0, 256, (plan["tune_count"], plan["buf_len"]), dtype=np.uint8)
        hops = list(range(plan["tune_count"]))
        _REF.update(kind="port", port=p, plan=plan, w=w, reads=reads, hops=hops,
                    per_pass=plan["tune_count"] * (plan["buf_len"] // 2))


def _ref_step(passes):
    """(seconds, samples, kind) for `passes` sweeps of the whole hop plan in this worker"""
    if _REF["kind"] == "reference":
        return _REF["ref"].scan_timed(passes), passes * _REF["per_pass"], "reference"
    t0 = time.perf_counter()
    for _ in range(passes):
        _REF["port"].scan(_REF["plan"], _REF["w"], _REF["reads"], _REF["hops"], _REF["plan"]["tune_count"])
    return time.perf_counter() - t0, passes * _REF["per_pass"], "port"


class CpuReference:
    """`procs` persistent worker processes, each an independent instance of the reference's
    single-threaded scanner() (the reference has no threads: rtl_power.c:29-36, 844-846)."""

    def __init__(self, procs, rng=RANGE, crop=CROP, window=WINDOW):
        import multiprocessing as mp
        self.procs = procs
        self.pool = mp.get_context("spawn").Pool(procs, initializer=_ref_init, initargs=(17, rng, crop, window))
        self.pool.map(_ref_step, [1] * procs)  # all workers up and configured

    def step(self, passes):
        res = self.pool.map(_ref_step, [passes] * self.procs, chunksize=1)
        return max(r[0] for r in res), sum(r[1] for r in res), res[0][2]

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    ref = CpuReference(cores)
    # bounded sample per step: the whole run stays within ~2 minutes whatever K is
    t_probe, s_probe, kind = ref.step(1)
    per_pass_s = max(t_probe, 1e-4)
    budget_s = 100.0
    passes = int(max(1, min(SWEEPS, budget_s / (args.steps + args.warmup) / per_pass_s)))
    for _ in range(args.warmup):
        ref.step(passes)
    total_t, total_s = 0.0, 0
    for _ in range(args.steps):
        t, smp, kind = ref.step(passes)
        total_t += t
        total_s += smp
    ref.close()
    value = total_s / total_t / 1e6
    sample = (f"{cores} independent processes x {passes} sweeps x 512 hops x 8192 samples per step "
              f"(of the {SWEEPS} sweeps of one step of the GPU arm)")
    line = {
        "metric": "input Msamples/s", "value": value, "unit": "Msamples/s", "impl": "reference",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int16/int64 fixed point", "data": "synthetic",
        "config": {"workload": WORKLOAD, "cli": f"-f {RANGE}", "hops": 512, "bins": 4096, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------- GPU arm

class Dist:
    """rank / world plumbing (torch.distributed over NCCL when N > 1)"""

    def __init__(self, torch, dist):
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        dev = "cuda" if self.dist.is_initialized() and self.dist.get_backend() == "nccl" else "cpu"
        t = self.torch.tensor([v], dtype=self.torch.float64, device=dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


class ShardedSweep:
    """One hop-sharded rtl_power scan: this rank's handle, its share of the synthetic input (pinned host
    copy + device-resident copy) and the per-interval exchange to rank 0."""

    def __init__(self, D, rs, rng, crop, window, fir, sweeps, peak=0, sizes=None, device_copy=True):
        import numpy as np
        from rtlsdr_b200.planner import plan_scan, synth_cube
        from rtlsdr_b200.sweep import SpectrumGather, shard_ranges
        torch = D.torch
        self.D, self.rs, self.np = D, rs, np
        self.plan = plan_scan(rng, crop, fir)
        pd = self.plan.as_dict()
        pd["peak_hold"] = peak
        self.pd, self.sweeps = pd, sweeps
        self.tc, self.b, self.n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
        self.sizes = [len(r) for r in shard_ranges(self.tc, D.world, sizes)]
        self.mine = shard_ranges(self.tc, D.world, sizes)[D.rank]
        self.h = len(self.mine)
        self.window = rs.window_coefs(window, self.n) if pd["bin_e"] else None
        # async_report: the report epilogue of interval k runs on the handle's report stream while the handle's own
        # stream already transforms interval k+1 into the second accumulator set
        self.g = rs.GpuScan.from_plan(pd, window_coefs=self.window, device=D.local, hops=list(self.mine), async_report=True)
        self.stream = torch.cuda.ExternalStream(self.g.get_stream())
        self.rstream = torch.cuda.ExternalStream(self.g.get_report_stream())
        self.gather = SpectrumGather(self.tc, self.n, self.g.db_count, D.world, D.rank, torch.device("cuda", D.local),
                                     sizes=sizes)
        self.bytes_rank = sweeps * self.h * self.b
        self.bytes_all = sweeps * self.tc * self.b
        # input: bytes of read (sweep p, hop) from the synthetic source, [sweeps, my hops, buf_len]
        self.pinned = rs.PinnedBuffer(self.bytes_rank)
        synth_cube(self.pinned.ptr, SYNTH_XORSHIFT, 0, 0, self.tc, self.mine.start, self.h, 0, sweeps, self.b)
        self.dev_in = None
        if device_copy:
            self.dev_in = torch.empty(self.bytes_rank, dtype=torch.uint8, device="cuda")
            self.dev_in.copy_(torch.from_numpy(self.pinned.array), non_blocking=False)
        self.extra = []     # second handle of the host-buffer leg

    def step_device(self, i, sweeps=None, to_host=False):
        k = i & 1
        self.g.submit_device(0, self.h, sweeps or self.sweeps, self.dev_in.data_ptr(), self.h * self.b, self.b)
        self.finish(self.g, self.rstream, k, to_host)

    def finish(self, g, rstream, k, to_host):
        """report epilogue into exchange buffer k (on the handle's report stream) + the exchange (asynchronous)"""
        self.gather.before_collect(k, rstream)
        g.collect_device(*self.gather.pointers(k))
        self.gather.publish(k, rstream, to_host=to_host)

    def report(self, k):
        """rank 0: IntervalReport of exchange buffer k; every rank blocks until the exchange is done"""
        return self.gather.fetch(k)

    def close(self):
        self.g.close()
        for g in self.extra:
            g.close()
        self.pinned.free()


def time_device(D, sw, steps, warmup, min_ms=MIN_TIMED_MS, sampler=None, last=None):
    """rounds of exactly `steps` device-resident steps, CUDA events on the launching stream, max over ranks;
    repeated until >= min_ms have been timed (min_ms = 0: one round).  Returns (ms_per_step, timed_steps, kernel_ms,
    kernel_launches, launches, issue_ms).  last: a list that receives rank 0's report of the last timed step."""
    torch = D.torch
    for i in range(warmup):
        sw.step_device(i)
    sw.stream.wait_stream(sw.rstream)
    sw.gather.drain(sw.stream)
    D.barrier()
    sw.g.kernel_time()      # arm / reset the per-kernel timers
    sw.g.set_timing(1)      # every transform launch is bracketed with events on the launching stream
    s0 = sw.g.stats()
    if sampler:
        sampler.start()
    total_ms, rounds, i0 = 0.0, 0, warmup
    want = 1
    issue_ms = 0.0      # host time to ISSUE one step (python + CUDA API calls): must stay below the GPU's step time
    while rounds < want:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record(sw.stream)
        t_issue = time.perf_counter()
        for i in range(steps):
            sw.step_device(i0 + i)
        issue_ms = max(issue_ms, 1e3 * (time.perf_counter() - t_issue) / steps)
        sw.stream.wait_stream(sw.rstream)   # the last reports ...
        sw.gather.drain(sw.stream)          # ... and exchanges are inside the timed region
        e1.record(sw.stream)
        D.barrier()
        ms = D.max(e0.elapsed_time(e1))
        total_ms += ms
        rounds += 1
        i0 += steps
        if rounds == 1:
            want = max(1, min(200, int(-(-min_ms // max(ms, 1e-3)))))
    s1 = sw.g.stats()
    k_ms, k_n = sw.g.kernel_time()
    sw.g.set_timing(0)
    if last is not None and D.rank == 0:
        # before the sampler's untimed launches below rewrite report buffer 0
        last.append(device_report(sw.gather, (i0 - 1) & 1))
    if sampler:
        # nvidia-smi ticks every 10 ms: keep the same kernels running on THIS rank, untimed and WITHOUT the
        # exchange (a collective that the other ranks do not join would never complete), until a few clock
        # samples exist
        t_end = time.perf_counter() + 1.0
        while len(sampler.rows) < 4 and time.perf_counter() < t_end:
            for _ in range(4):
                sw.g.submit_device(0, sw.h, sw.sweeps, sw.dev_in.data_ptr(), sw.h * sw.b, sw.b)
                sw.g.collect_device(*sw.gather.pointers(0))
            torch.cuda.synchronize()
    return (total_ms / (rounds * steps), rounds * steps, k_ms / max(k_n, 1), k_n,
            s1["kernel_launches"] - s0["kernel_launches"], D.max(issue_ms))


def device_report(gather, k):
    """rank 0, after a synchronise: the gathered report in exchange buffer k where the device left it (timed steps
    publish without the copy to pinned host memory that fetch() reads)"""
    bufs = gather.send[k].view(1, gather.words) if gather.world == 1 else gather.recv[k]
    return gather.unpack(bufs.cpu().numpy())


def dump_outputs(path, rep):
    """avg (int64 bins, exact in float64 below 2^53), db and samples of one report as float64 .npy files"""
    import numpy as np
    assert int(np.abs(rep.avg).max()) < 1 << 53, "bins beyond float64's exact integers"
    os.makedirs(path, exist_ok=True)
    for name in ("avg", "db", "samples"):
        np.save(os.path.join(path, f"{name}.npy"), getattr(rep, name).astype(np.float64))


def verify_sharded(D, sw, kat_p1, full_interval=True):
    """Outside any timed region.  (a) sweep 0 alone, gathered over all ranks, FNV == the reference-generated
    known-answer hash; (b) the whole interval, gathered, FNV == a 1-rank run of the same bytes on rank 0."""
    from rtlsdr_b200.planner import fnv1a_int64, synth_cube
    np, rs, torch = sw.np, sw.rs, D.torch
    out = {}
    sw.step_device(0, sweeps=1, to_host=True)
    rep = sw.report(0)
    if D.rank == 0:
        got = fnv1a_int64(rep.avg)
        out.update(kat_sweeps=1, kat_fnv=f"{got:016x}", kat_expected=f"{kat_p1:016x}",
                   kat_ok=bool(got == kat_p1 and (rep.samples == 2).all()),
                   kat_source="SURVEY.md 8(c): unmodified rtl_power.c, same range, 1 sweep, xorshift source")
    if full_interval:
        sw.step_device(1, to_host=True)
        rep = sw.report(1)
        if D.rank == 0:
            got = fnv1a_int64(rep.avg)
            out.update(interval_sweeps=sw.sweeps, interval_fnv=f"{got:016x}", interval_ranks=D.world)
            if D.world == 1:
                # second, differently batched pass over the same bytes: four submits of a quarter interval each
                q = sw.sweeps // 4
                for c in range(4):
                    sw.g.submit_device(0, sw.h, q, sw.dev_in.data_ptr() + c * q * sw.h * sw.b, sw.h * sw.b, sw.b)
                avg1, smp1, _ = sw.g.collect_all(want_db=False)
                out["interval_fnv_check"] = f"{fnv1a_int64(avg1):016x}"
                out["interval_check"] = "same handle, interval re-submitted as 4 quarter batches + collect_all (host copy)"
                out["interval_ok"] = bool(fnv1a_int64(avg1) == got and (smp1 == rep.samples).all())
            else:
                # 1-rank run of the same bytes: rank 0 regenerates ALL hops' reads and scans them alone
                g1 = rs.GpuScan.from_plan(sw.pd, window_coefs=sw.window, device=D.local)
                hb = rs.PinnedBuffer(sw.bytes_all)
                synth_cube(hb.ptr, SYNTH_XORSHIFT, 0, 0, sw.tc, 0, sw.tc, 0, sw.sweeps, sw.b)
                g1.submit_batch(0, sw.tc, sw.sweeps, hb.ptr, sw.tc * sw.b, sw.b)
                avg1, smp1, _ = g1.collect_all(want_db=False)
                g1.close()
                hb.free()
                one = fnv1a_int64(avg1)
                out["interval_fnv_check"] = f"{one:016x}"
                out["interval_check"] = "1-rank run of the same bytes on rank 0 (all hops regenerated from the synthetic source)"
                out["interval_ok"] = bool(one == got and (smp1 == rep.samples).all())
    D.barrier()
    if D.rank == 0:
        out["ok"] = bool(out.get("kat_ok") and out.get("interval_ok", True))
    return out


def time_e2e(D, sw, steps, warmup):
    """The interval through the host-buffer ABI: pinned host input -> submit_batch (H2D) -> transform ->
    report epilogue -> exchange -> rank 0 copies the gathered report to host memory.  Two handles alternate,
    so interval i+1 crosses PCIe while interval i is transformed and exchanged (what a continuously
    running rtl_power does).  Wall clock between barriers, max over ranks."""
    torch, rs = D.torch, sw.rs
    g2 = rs.GpuScan.from_plan(sw.pd, window_coefs=sw.window, device=D.local, hops=list(sw.mine), async_report=True)
    sw.extra.append(g2)
    handles = [(sw.g, sw.rstream), (g2, torch.cuda.ExternalStream(g2.get_report_stream()))]

    def submit(i):
        handles[i & 1][0].submit_batch(0, sw.h, sw.sweeps, sw.pinned.ptr, sw.h * sw.b, sw.b)

    def run(n):
        submit(0)
        rep = None
        for i in range(n):
            if i + 1 < n:
                submit(i + 1)
            g, st = handles[i & 1]
            sw.finish(g, st, i & 1, True)
            rep = sw.report(i & 1)
        return rep

    run(max(2, min(warmup, 4)))
    D.barrier()
    t0 = time.perf_counter()
    rep = run(steps)
    torch.cuda.synchronize()
    dt = D.max(time.perf_counter() - t0)
    if D.rank == 0:
        assert int(rep.samples[0]) == 2 * sw.sweeps and int(rep.samples[-1]) == 2 * sw.sweeps, \
            "e2e report does not cover one whole interval"
    return dt, rep


def probe_h2d(D):
    """host-to-device GB/s of every rank's GPU with ALL ranks copying at the same time (pinned memory, CUDA events):
    the GPUs of one box do not all see the same host bandwidth (profiles/r02i_pcie_topo_8gpu.json)"""
    torch = D.torch
    nbytes = 128 << 20
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        dev.copy_(host, non_blocking=True)
    st.synchronize()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        e0.record(st)
        for _ in range(6):
            dev.copy_(host, non_blocking=True)
        e1.record(st)
    st.synchronize()
    gbs = 6 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    if D.world == 1:
        return [gbs]
    dev_t = "cuda" if D.dist.get_backend() == "nccl" else "cpu"
    mine = torch.tensor([gbs], dtype=torch.float64, device=dev_t)
    every = [torch.zeros(1, dtype=torch.float64, device=dev_t) for _ in range(D.world)]
    D.dist.all_gather(every, mine)
    return [float(t.item()) for t in every]


class ReadShardedSweep:
    """A scan with fewer hops than GPUs (BASELINE configs[3]: ONE hop of 2^17 bins, peak hold): the READS of every
    interval are dealt to the ranks, every rank's epilogue stores its raw int64 bins + counts into its slot of rank
    0's buffer (same exchange as the hop-sharded report), rank 0 folds the slots into its own handle
    (rtlsdr_gpu_scan_merge_device: sums / peak-hold maxima, exact) and writes the final report."""

    def __init__(self, D, rs, rng, window, peak, reads):
        import numpy as np
        from rtlsdr_b200.planner import plan_scan, synth_cube
        from rtlsdr_b200.sweep import SpectrumGather, shard_hops
        torch = D.torch
        self.D, self.rs, self.np = D, rs, np
        pd = plan_scan(rng, 0.0, None).as_dict()
        pd["peak_hold"] = peak
        self.pd, self.reads = pd, reads
        self.tc, self.b, self.n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
        self.mine = shard_hops(reads, D.world, D.rank)            # contiguous share of the interval's sweeps
        self.window = rs.window_coefs(window, self.n)
        # async_report: the epilogue that stores this rank's raw bins runs on the handle's report stream while its own
        # stream already transforms the next interval into the second accumulator set.  Rank 0 merges and reports
        # with a SECOND handle on that handle's stream, so nothing of the exchange sits on a transform stream.
        self.g = rs.GpuScan.from_plan(pd, window_coefs=self.window, device=D.local, async_report=True)
        self.stream = torch.cuda.ExternalStream(self.g.get_stream())
        self.rstream = torch.cuda.ExternalStream(self.g.get_report_stream())
        self.g_merge = rs.GpuScan.from_plan(pd, window_coefs=self.window, device=D.local) if D.rank == 0 else None
        self.mstream = torch.cuda.ExternalStream(self.g_merge.get_stream()) if self.g_merge else None
        self.gather = SpectrumGather(self.tc, self.n, self.g.db_count, D.world, D.rank, torch.device("cuda", D.local),
                                     mode=("host" if os.environ.get("BENCH_GLOO_ONE_GPU") and D.world > 1 else None),
                                     replicated=True)
        self.bytes_all = reads * self.tc * self.b
        nb = max(1, len(self.mine) * self.tc * self.b)
        pinned = rs.PinnedBuffer(nb)
        if len(self.mine):
            synth_cube(pinned.ptr, SYNTH_XORSHIFT, 0, 0, self.tc, 0, self.tc, self.mine.start, len(self.mine), self.b)
        self.dev_in = torch.empty(nb, dtype=torch.uint8, device="cuda")
        self.dev_in.copy_(torch.from_numpy(pinned.array), non_blocking=False)
        pinned.free()
        self.out = torch.zeros(self.tc * (self.n + self.g.db_count + 1), dtype=torch.int64, device="cuda") \
            if D.rank == 0 else None

    def step(self, i):
        k = i & 1
        if len(self.mine):
            self.g.submit_device(0, self.tc, len(self.mine), self.dev_in.data_ptr(), self.tc * self.b, self.b)
        self.gather.before_collect(k, self.rstream)
        p_avg, p_smp, _ = self.gather.pointers(k)
        self.g.collect_device(p_avg, p_smp, None)
        self.gather.publish(k, self.rstream)
        if self.D.rank == 0:
            self.mstream.wait_event(self.gather.gathered[k])
            self.g_merge.merge_device(*self.gather.partial_sets(k))
            self.gather.release_copy(k, self.mstream)
            base = self.out.data_ptr()
            p_db = base + self.tc * self.n * 8
            self.g_merge.collect_device(base, p_db + self.tc * self.g.db_count * 8, p_db)

    def drain(self):
        """the handle's stream waits for every report, exchange and merge issued so far"""
        self.stream.wait_stream(self.rstream)
        self.gather.drain(self.stream)
        if self.mstream is not None:
            self.stream.wait_stream(self.mstream)

    def merged_bins(self):
        self.D.torch.cuda.synchronize()
        return self.out[: self.tc * self.n].cpu().numpy().reshape(self.tc, self.n)

    def close(self):
        self.g.close()
        if self.g_merge:
            self.g_merge.close()


def read_sharded_companion(D, rs, steps, peak_gbs):
    """N > 1: BASELINE configs[3] with 8 x 256 reads per interval dealt to the ranks (strong scaling of one job);
    the merged bins of one interval are verified against a 1-rank scan of the same bytes on rank 0."""
    from rtlsdr_b200.planner import fnv1a_int64, synth_cube
    from rtlsdr_b200.sweep import shard_hops
    torch = D.torch
    rng, window, reads = "100M:102.4M:19", "blackman-harris", 2048
    sw = ReadShardedSweep(D, rs, rng, window, 1, reads)
    out = {"workload": "large_fft_2^17_blackman-harris_peak_hold (BASELINE configs[3]), READS sharded over the GPUs, "
                       "raw accumulators merged on rank 0 (rtlsdr_gpu_scan_merge_device)",
           "cli": f"-f {rng} -P", "reads_per_interval": reads,
           "reads_per_gpu": [len(shard_hops(reads, D.world, r)) for r in range(D.world)], "unit": "Msamples/s",
           "exchange": sw.gather.describe()}
    # ---- verification (outside the timed region): one full interval vs a 1-rank scan of ALL its bytes on rank 0
    sw.step(0)
    got = sw.merged_bins() if D.rank == 0 else None
    if D.rank == 0:
        g1 = rs.GpuScan.from_plan(sw.pd, window_coefs=sw.window, device=D.local)
        chunk = 256
        hb = rs.PinnedBuffer(chunk * sw.tc * sw.b)
        for lo in range(0, reads, chunk):
            synth_cube(hb.ptr, SYNTH_XORSHIFT, 0, 0, sw.tc, 0, sw.tc, lo, chunk, sw.b)
            g1.submit_batch(0, sw.tc, chunk, hb.ptr, sw.tc * sw.b, sw.b)
            g1.sync()
        avg1, _, _ = g1.collect_all(want_db=False)
        g1.close()
        hb.free()
        out["verify"] = {"ok": bool(fnv1a_int64(avg1) == fnv1a_int64(got)), "fnv": f"{fnv1a_int64(got):016x}",
                         "check": "merged bins of the read-sharded interval == a 1-rank scan of the same 2048 reads on rank 0"}
    D.barrier()
    for i in range(3):
        sw.step(1 + i)
    sw.drain()
    D.barrier()
    total, done, want, rounds = 0.0, 0, 1, 0
    while rounds < want:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record(sw.stream)
        for i in range(steps):
            sw.step(4 + done + i)
        sw.drain()
        e1.record(sw.stream)
        D.barrier()
        ms = D.max(e0.elapsed_time(e1))
        total += ms
        done += steps
        rounds += 1
        if rounds == 1:
            want = max(1, min(50, int(-(-MIN_TIMED_MS // max(ms, 1e-3)))))
    sw.close()
    ms = total / done
    out.update(value=sw.bytes_all / 2 / (ms * 1e-3) / 1e6, ms_per_step=ms, timed_steps=done, bytes_per_step=sw.bytes_all,
               frac_of_hbm_peak=sw.bytes_all / (ms * 1e-3) / 1e9 / (peak_gbs * D.world))
    return out


def companion(rs, plan_scan, torch, name, freq, crop, window, fir, peak, passes, steps, peak_gbs):
    """Device-resident throughput of another rtl_power configuration on one GPU (same method as `value`)."""
    plan = plan_scan(freq, crop, fir)
    pd = plan.as_dict()
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
    total, done = 0.0, 0
    while total < MIN_TIMED_MS and done < 200 * steps:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            step(3 + done + i)
        e1.record(stream)
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
        done += steps
    ms = total / done
    g.close()
    del dev_in
    gbs = step_bytes / (ms * 1e-3) / 1e9
    return {"workload": name, "cli": f"-f {freq}" + (f" -F {fir}" if fir is not None else "") + (" -P" if peak else ""),
            "plan": {k: pd[k] for k in ("tune_count", "bin_e", "buf_len", "downsample", "downsample_passes")},
            "value": step_bytes / 2 / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms, "timed_steps": done,
            "bytes_per_step": step_bytes, "achieved_GBps": gbs, "frac_of_hbm_peak": gbs / peak_gbs}


def run_gpu(args):
    import torch
    import torch.distributed as dist

    import rtlsdr_b200.scan as rs
    from rtlsdr_b200.planner import plan_scan
    from rtlsdr_b200.sweep import shard_hops

    D = Dist(torch, dist)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback")
    one_gpu = bool(os.environ.get("BENCH_GLOO_ONE_GPU"))   # tests: every rank on cuda:0, reports exchanged through gloo
    if one_gpu:
        D.local = 0
    torch.cuda.set_device(D.local)
    pin = pin_to_gpu_numa(D.local)            # before any pinned allocation
    if D.world > 1:
        if one_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", D.local))
    rs.load_library()
    peak, peak_src = read_peaks()

    # ---- headline: BASELINE configs[4], hops sharded over the ranks ----
    sw = ShardedSweep(D, rs, RANGE, CROP, WINDOW, FIR, args.sweeps)
    verify = verify_sharded(D, sw, KAT_P1)
    sampler = ClockSampler(D.local) if D.rank == 0 else None
    last = []
    ms_step, timed_steps, k_ms, k_n, launches, issue_ms = time_device(D, sw, args.steps, args.warmup, min_ms=0.0,
                                                                      sampler=sampler, last=last)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    # ---- end to end from host buffers: hop shares proportional to each GPU's host-to-device bandwidth ----
    e2e_steps = max(4, min(args.steps, 24))
    h2d = probe_h2d(D)
    forced = os.environ.get("BENCH_E2E_WEIGHTS")           # tests
    weights = [float(x) for x in forced.split(",")] if forced else h2d
    sw_e2e, e2e_shares = sw, "equal"
    if D.world > 1 and len(weights) == D.world and max(weights) > 1.1 * min(weights):
        from rtlsdr_b200.sweep import weighted_sizes
        sizes = weighted_sizes(sw.tc, weights)
        sw_e2e = ShardedSweep(D, rs, RANGE, CROP, WINDOW, FIR, args.sweeps, sizes=sizes, device_copy=False)
        e2e_shares = "proportional to the measured host-to-device bandwidth of every GPU"
    e2e_s, e2e_rep = time_e2e(D, sw_e2e, e2e_steps, args.warmup)
    e2e_ok = None
    if D.rank == 0:
        from rtlsdr_b200.planner import fnv1a_int64
        e2e_ok = bool(f"{fnv1a_int64(e2e_rep.avg):016x}" == verify.get("interval_fnv"))
    e2e_sizes = list(sw_e2e.sizes)
    e2e_d2h = sw_e2e.gather.world * sw_e2e.gather.words * 8
    if sw_e2e is not sw:
        sw_e2e.close()

    # ---- second sharded workload: BASELINE configs[2] (623 hops do not divide evenly) ----
    sw3 = ShardedSweep(D, rs, RANGE3, 0.0, "rectangle", FIR3, max(1, SWEEPS3 * args.sweeps // SWEEPS))
    verify3 = verify_sharded(D, sw3, KAT3_P1, full_interval=False)
    ms3, steps3, k3_ms, _, _, _ = time_device(D, sw3, max(4, min(args.steps, 20)), 3)
    comp3 = None
    if D.rank == 0:
        v3 = sw3.bytes_all / 2 / (ms3 * 1e-3) / 1e6
        comp3 = {"workload": "wideband_sweep_24-1766MHz_623_hops_4096bins_64_sweeps (BASELINE configs[2]), hops sharded",
                 "cli": f"-f {RANGE3} -F {FIR3}", "value": v3, "unit": "Msamples/s", "ms_per_step": ms3,
                 "timed_steps": steps3, "hops_per_gpu": [len(shard_hops(sw3.tc, D.world, r)) for r in range(D.world)],
                 "bytes_per_step": sw3.bytes_all, "frac_of_hbm_peak": sw3.bytes_all / (ms3 * 1e-3) / 1e9 / (peak * D.world),
                 "verify": verify3}
    sw3.close()
    # ---- N > 1: a single-hop scan (BASELINE configs[3]) with its READS sharded and an exact merge on rank 0 ----
    comp4 = None
    if D.world > 1 and not args.no_companions:
        comp4 = read_sharded_companion(D, rs, max(4, min(args.steps, 20)), peak)

    if D.rank == 0:
        samples_step = sw.bytes_all // 2
        value = samples_step / (ms_step * 1e-3) / 1e6
        e2e = samples_step * e2e_steps / e2e_s / 1e6
        achieved = sw.bytes_rank / (k_ms * 1e-3) / 1e9 if k_n else None
        ncu = read_ncu()
        traffic = ncu.get("dram_bytes_per_launch") if ncu.get("launch_bytes") == sw.bytes_rank else None
        d2h = e2e_d2h
        line = {
            "metric": "input Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": D.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "timed_steps": timed_steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int16/int64 fixed point", "data": "synthetic",
            "config": {"workload": WORKLOAD if sw.sweeps == SWEEPS else
                       f"REDUCED TEST SIZE ({sw.sweeps} sweeps per step, not a benchmark result) of {WORKLOAD}",
                       "cli": f"-f {RANGE}", "hops": sw.tc, "bins": sw.n,
                       "sweeps_per_step": sw.sweeps, "reads_per_step": sw.sweeps * sw.tc, "bytes_per_step": sw.bytes_all,
                       "hops_per_gpu": [len(shard_hops(sw.tc, D.world, r)) for r in range(D.world)],
                       "input": "synthetic source xorshift stream, bytes a pure function of (hop, sweep): "
                                "identical job at every N",
                       "cache": f"inputs larger than L2: every step streams this rank's whole {sw.bytes_rank >> 20} MiB cube from HBM",
                       "timing": f"{timed_steps} steps between two CUDA events",
                       "exchange": sw.gather.describe(), "host_pinning": pin},
            "per_gpu_value": value / D.world,
            "host_issue_ms_per_step": issue_ms,
            "verify": verify,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "traffic_source": ncu.get("source") if traffic else None,
                         "kernel": "scan_small_kernel<12,0,0>", "kernel_ms": k_ms, "kernel_launches_timed": k_n,
                         "kernel_timing": "CUDA events on the launching stream around every transform launch of the timed region (rank 0)",
                         "algorithmic_bytes_per_launch": sw.bytes_rank, "peak_source": peak_src,
                         "note": "integer-issue bound, not HBM bound at ds = 1: see DESIGN.md; roofline.issue is the bound it runs against"},
            "e2e": {"value": e2e, "unit": "Msamples/s", "h2d_bytes_per_step": sw.bytes_all,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "hop_shares": e2e_shares, "hops_per_gpu": e2e_sizes,
                    "h2d_GBps_per_gpu_all_copying": [round(x, 1) for x in h2d],
                    "report_fnv_equals_verified_interval": e2e_ok,
                    "api": "rtlsdr_gpu_scan_submit_batch (pinned host input, every rank its hops) + report epilogue + "
                           "exchange + gathered report copied to pinned host memory on rank 0; two handles alternate "
                           "so the next interval's copies overlap the transform"},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if k_n and clocks and clocks.get("sm_mhz") and ncu.get("warp_instructions_per_byte"):
            sms = torch.cuda.get_device_properties(0).multi_processor_count
            inst = ncu["warp_instructions_per_byte"] * sw.bytes_rank
            ipc = inst / (k_ms * 1e-3 * clocks["sm_mhz"] * 1e6 * sms)
            pk = ncu["issue_peak_warp_instr_per_clk_per_sm"]
            line["roofline"]["issue"] = {"bound": "issue", "achieved": ipc, "peak": pk, "unit": "warp-instr/clk/SM",
                                         "frac": ipc / pk, "warp_instructions_per_launch": inst,
                                         "sm_mhz": clocks["sm_mhz"], "sms": sms, "peak_source": ncu.get("issue_peak_source")}
        comps = [comp3] + ([comp4] if comp4 else [])
        if D.world == 1 and not args.no_companions:
            try:
                comps += [
                    companion(rs, plan_scan, torch, "fm_band_scan_88-108MHz_4096bins_hamming_crop20_10s (BASELINE configs[1], "
                              "round 1's headline)", RANGE2, CROP2, WINDOW2, None, 0, SWEEPS2, 50, peak),
                    companion(rs, plan_scan, torch, "single_hop_2.4MSps_1024bins_rectangle_1s (BASELINE configs[0])",
                              "100M:102.4M:2400", 0.0, "rectangle", None, 0, 293, 50, peak),
                    companion(rs, plan_scan, torch, "narrow_scan_boxcar_ds28_1024bins", "100M:100.1M:100", 0.0,
                              "rectangle", None, 0, 8192, 10, peak),
                    companion(rs, plan_scan, torch, "rms_1MHz_bins_10hops", "100M:110M:1M", 0.0,
                              "rectangle", None, 0, 4096, 10, peak),
                    companion(rs, plan_scan, torch, "narrow_scan_fifth_order_x4_fir9_1024bins", "100M:100.1M:100", 0.0,
                              "blackman", 9, 0, 8192, 10, peak),
                    companion(rs, plan_scan, torch, "large_fft_2^17_blackman-harris_peak_hold (BASELINE configs[3])",
                              "100M:102.4M:19", 0.0, "blackman-harris", None, 1, 256, 10, peak),
                ]
            except Exception as exc:  # companions are extra evidence, never fail the bench line
                comps.append({"error": repr(exc)})
        line["companions"] = comps
        if D.world == 1 and not args.no_cpu:
            ref = CpuReference(1)
            t, smp, kind = ref.step(100)
            ref.close()
            line["cpu_baseline"] = {"value": smp / t / 1e6, "unit": "Msamples/s", "cores": 1, "kind": kind,
                                    "sample": "100 sweeps x 512 hops x 8192 samples (419 M samples) of the same workload, 1 thread"}
        print(json.dumps(line))
    sw.close()
    ok = True
    if D.rank == 0:
        ok = bool(verify.get("ok")) and bool(verify3.get("ok")) and e2e_ok is not False
        if not ok:
            print("bench.py: VERIFY FAILED: gathered bins differ from the known answer / the 1-rank run", file=sys.stderr)
    if D.world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0 if ok else 1


def pin_to_gpu_numa(gpu_index):
    """Bind this process to the CPUs (and so, by first touch, the memory) of the NUMA node its GPU hangs off,
    before any pinned allocation (VERDICT r1 weak #5).  Returns a description for the bench line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node"
        node = int(open(path).read().strip()) if os.path.exists(path) else -1
        if node < 0:
            return {"numa_node": node, "bound": False, "why": "no NUMA affinity reported for the GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return {"numa_node": node, "bound": False, "why": "node CPUs not in this process's affinity mask"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "bound": True, "cpus": f"{allowed[0]}-{allowed[-1]} ({len(allowed)})"}
    except Exception as exc:  # noqa: BLE001 -- best effort
        return {"bound": False, "why": repr(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of the headline workload")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--sweeps", type=int, default=SWEEPS,
                    help="sweeps per step (default = the benchmark's 256; tests shrink it, the line says so)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-companions", action="store_true", help="skip the other-configuration measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's report of the last timed step to DIR/{avg,db,samples}.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
