"""Hop-sharded rtl_power sweep over the GPUs of one box (SURVEY.md 8e).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        -m rtlsdr_b200.sweep_main -f 24M:1766M:1k --sweeps 6 --intervals 2 -o scan.csv

Every rank plans the same scan (host/rtl_power_plan.c), takes a contiguous range of hops
(`shard_hops`), drives its own rtlsdr_gpu_scan handle from the synthetic source (bytes are a pure
function of (hop, sweep), so the result does not depend on N), and once per integration interval
bins + dB rows + sample counts reach rank 0 -- written by every rank's report epilogue straight
into rank 0's buffer over NVLink (symmetric-memory peer mapping, one barrier per interval), or by
ONE NCCL gather where peer mapping is unavailable / RTLSDR_B200_NCCL_GATHER=1 -- and rank 0 formats
the reference's CSV rows in hop order (rtl_power.c:995-1000) on its GPU (rtlsdr_gpu_scan_format_csv_device, once
per rank slot) and copies only the text to the host.  With N = 1 no process group is created.
Scans with fewer hops than GPUs (BASELINE configs 1 and 4 are ONE hop) shard the READS instead (--shard reads):
every rank transforms its share of each hop's reads into its own accumulators, the raw int64 bins and counts
reach rank 0 the same way, and rank 0 folds them into its handle (rtlsdr_gpu_scan_merge_device: int64 sums, or
maxima under -P, are associative and exact) before its ordinary collect -- rows byte-identical to one GPU's.
Hop order inside a rank's shard can be randomised (--random-hops SEED, the reference's TODO list
rtl_power.c:29-36): the bins are order independent (int64 sums / maxima, rtl_power.c:708-716).
--sk FILE also writes every bin's spectral kurtosis (RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS): rows with the power rows'
prefix and %.4f values (nan where undefined), the bytes rtl_power_gpu -K writes.  Hop-sharded, every rank's
collect_sk_device() adds its SK rows to its report slot and rank 0 formats them beside the power rows
(rtlsdr_gpu_scan_format_sk_csv_device); read-sharded, the slots also carry S2 (the exact 128-bit sums of |X|^4) and
rank 0 folds all three sums into its handle (rtlsdr_gpu_scan_merge_sk_device) before rtlsdr_gpu_scan_collect_sk_csv
-- SK rows byte-identical to one GPU's.  The power CSV is the same with and without --sk.  Not with -P or 1-bin
(rms) hops.
--excise FILE writes the spectral-kurtosis-excised power rows (RTLSDR_GPU_FLAG_SK_EXCISION, hop-sharded only): every
interval's sweeps are submitted in chunks of --excise-sweeps K passes with rtlsdr_gpu_scan_excise_fold() after each
chunk, so a bin's sub-integration of K sweeps enters its clean average only when its SK lies within
[1 - LOW sigma, 1 + HIGH sigma] (--excise-sigma LOW[:HIGH], default 3:3, inf never flags that side).  Every rank's
excised_report_device() adds the excised dB rows, the flag fractions and the folded sample counts to its report slot
(SpectrumGather(excise=True)) in front of its collect_sk_device(); rank 0 formats them like the power rows
(--excise) and like the SK rows (--excise-flags FILE), with the folded samples as the count column.  The power and
SK files are the same with and without --excise.  Not with --shard reads (merged reads would land in one
sub-integration), -P or 1-bin hops.
"""
import argparse
import ctypes
import os
import sys

import numpy as np


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("-f", dest="range", required=True, help="lower:upper:bin_size (like rtl_power)")
    ap.add_argument("-c", dest="crop", default="0", help="crop percent, e.g. 20%%")
    ap.add_argument("-w", dest="window", default="rectangle")
    ap.add_argument("-F", dest="fir", type=int, default=None)
    ap.add_argument("-P", dest="peak", action="store_true")
    ap.add_argument("--sweeps", type=int, default=8, help="sweeps over all hops per integration interval")
    ap.add_argument("--intervals", type=int, default=1)
    ap.add_argument("--synth", default="xorshift", choices=["xorshift", "counter", "const", "biased", "tone"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--param", type=int, default=0)
    ap.add_argument("--stamp", default="2026-01-01, 00:00:00", help="fixed 'date, time' prefix of the rows")
    ap.add_argument("--random-hops", type=int, default=None, metavar="SEED",
                    help="visit the hops of every sweep in a random order (results do not depend on it)")
    ap.add_argument("--shard", default="hops", choices=["hops", "reads"],
                    help="hops: contiguous hop ranges per GPU (default); reads: every GPU takes a share of the sweeps "
                         "of ALL hops and rank 0 merges the raw accumulators (single-hop scans)")
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"],
                    help="gloo: reports are staged through host memory (e.g. several ranks on one GPU in tests)")
    ap.add_argument("--device", type=int, default=None, help="CUDA device of this rank (default: LOCAL_RANK)")
    ap.add_argument("--sk", dest="sk_out", default=None, metavar="FILE",
                    help="also write each bin's spectral kurtosis to FILE (rows like the power rows, %%.4f values)")
    ap.add_argument("--excise", dest="excise_out", default=None, metavar="FILE",
                    help="also write the spectral-kurtosis-excised power rows to FILE (sub-integrations whose SK lies "
                         "outside the thresholds are left out of a bin's average)")
    ap.add_argument("--excise-flags", dest="flags_out", default=None, metavar="FILE",
                    help="with --excise: the flagged fraction of every bin's sub-integrations (%%.4f values)")
    ap.add_argument("--excise-sweeps", type=int, default=None, metavar="K",
                    help="with --excise: sweeps per sub-integration (default: the fewest giving every hop 64 FFT "
                         "blocks)")
    ap.add_argument("--excise-sigma", default="3:3", metavar="LOW[:HIGH]",
                    help="with --excise: thresholds 1 - LOW*sigma and 1 + HIGH*sigma (default 3:3)")
    ap.add_argument("--guard-bits", action="store_true",
                    help="fix_fft with 8 fractional guard bits (RTLSDR_GPU_FLAG_GUARD_BITS): the transform rounds "
                         "2^8 below the reference's LSB, so fine-resolution rows show the signal's noise floor")
    ap.add_argument("-o", dest="out", default="-")
    args = ap.parse_args(argv)
    if args.sk_out is not None and args.peak:
        raise SystemExit("sweep_main: --sk needs averaged power bins, not -P peak hold")
    excise = args.excise_out is not None
    k_low = k_high = None
    if args.flags_out is not None and not excise:
        raise SystemExit("sweep_main: --excise-flags needs --excise")
    if excise:
        if args.shard == "reads":
            raise SystemExit("sweep_main: --excise needs all reads of a hop on one rank, not --shard reads")
        if args.peak:
            raise SystemExit("sweep_main: --excise needs averaged power bins, not -P peak hold")
        if args.excise_sweeps is not None and args.excise_sweeps < 1:
            raise SystemExit("sweep_main: --excise-sweeps must be >= 1")
        try:
            lo, _, hi = args.excise_sigma.partition(":")
            k_low, k_high = float(lo), float(hi or lo)
        except ValueError:
            k_low = k_high = float("nan")
        if not (k_low >= 0 and k_high >= 0):
            raise SystemExit("sweep_main: --excise-sigma LOW[:HIGH] needs two values >= 0")

    import torch
    import torch.distributed as dist

    from . import scan as rs
    from .planner import host_library, plan_scan, synth_cube
    from .sweep import SpectrumGather, shard_hops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0")) if args.device is None else args.device
    if not torch.cuda.is_available():
        raise SystemExit("sweep_main: no CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        if args.backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")

    host = host_library()
    crop = host.rp_atofp(args.crop.encode())
    plan = plan_scan(args.range, crop, args.fir)
    pd = plan.as_dict()
    pd["peak_hold"] = 1 if args.peak else 0
    sk = args.sk_out is not None
    if sk and pd["bin_e"] == 0:
        raise SystemExit("sweep_main: --sk needs FFT bins; this scan's hops are 1-bin (rms) power readings")
    if excise and pd["bin_e"] == 0:
        raise SystemExit("sweep_main: --excise needs FFT bins; this scan's hops are 1-bin (rms) power readings")
    if args.guard_bits and pd["bin_e"] == 0:
        raise SystemExit("sweep_main: --guard-bits needs FFT bins; this scan's hops are 1-bin (rms) power readings")
    sk = sk or excise          # an excision handle is an SK handle: its report is collect_sk_device()
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    mine = shard_hops(tc, world, rank)
    mode = ["xorshift", "counter", "const", "biased", "tone"].index(args.synth)
    if args.shard == "reads":
        return _main_read_sharded(args, rs, host, plan, pd, mode, world, rank, local, torch, dist,
                                  SpectrumGather, shard_hops, synth_cube)

    g = None
    if len(mine):
        window = rs.window_coefs(args.window, n) if pd["bin_e"] else None
        g = rs.GpuScan.from_plan(pd, window_coefs=window, device=local, hops=list(mine), spectral_kurtosis=sk,
                                 guard_bits=args.guard_bits, sk_excision=excise)
    # sub-integration length: K passes per fold (the same K on every rank: FFT blocks per read do not depend on the hop)
    chunk = (args.excise_sweeps or g.excise_sweeps()) if (g and excise) else args.sweeps
    db_count = g.db_count if g else plan.db_count
    gather = SpectrumGather(tc, n, db_count, world, rank, torch.device("cuda", local),
                            mode=("host" if args.backend == "gloo" and world > 1 else None), sk=sk, excise=excise)
    if rank == 0 and world > 1:
        print("sweep_main: interval reports: " + gather.describe(), file=sys.stderr)
    stream = torch.cuda.ExternalStream(g.get_stream()) if g else torch.cuda.current_stream()
    stamp = args.stamp + ", "
    groups = ["power"] + (["sk"] if args.sk_out is not None else []) + (["excise"] if excise else []) + \
        (["flags"] if args.flags_out is not None else [])
    if rank == 0:
        # rank 0 formats every rank's rows from a private device copy of the gathered report, on its handle's
        # stream behind the exchange; one text region and one int64 length per rank slot, copied out together
        gather.keep_device_copy()
        g.set_csv_columns(*plan.csv_columns())
        # one text region per (output, rank slot): the power rows, then with --sk the SK rows, with --excise the
        # excised rows and, with --excise-flags, the flag rows; group gi's regions are slots gi*world..gi*world+world-1
        caps = []
        for name in groups:
            cap = g.sk_csv_capacity if name in ("sk", "flags") else g.csv_capacity
            caps += [cap(len(r), len(stamp.encode())) for r in gather.ranges]
        offs = [0] + [int(x) for x in np.cumsum(caps)]
        lens_at = (offs[-1] + 7) // 8 * 8
        dev = torch.device("cuda", local)
        text_dev = [torch.empty(lens_at + 8 * len(caps), dtype=torch.uint8, device=dev) for _ in range(2)]
        text_host = [torch.empty(lens_at + 8 * len(caps), dtype=torch.uint8).pin_memory() for _ in range(2)]
        text_ready = [torch.cuda.Event() for _ in range(2)]
    # Two pinned input cubes alternate: rtlsdr_gpu_scan_submit_batch() returns while its host-to-device copies
    # are still queued, and `buf` must stay untouched until an event recorded on the handle's stream after the
    # call has completed (include/rtlsdr_gpu_scan.h) -- `consumed[k]` below.
    pinned = [rs.PinnedBuffer(max(1, args.sweeps * len(mine) * b)) for _ in range(2)] if g else None
    consumed = [None, None]

    rng = np.random.default_rng(args.random_hops + 7919 * rank) if args.random_hops is not None else None
    outs = {name: [] for name in groups}
    pending = None          # exchange buffer of the interval whose report has not been printed yet

    def format_rows(k):
        """rank 0: the rows of exchange buffer k into text_dev[k] on the handle's stream, then to pinned memory"""
        stream.wait_event(gather.gathered[k])
        lens = text_dev[k].data_ptr() + lens_at
        for r, hops in enumerate(gather.ranges):
            if len(hops):
                p_db, p_smp = gather.slot_rows(k, r)
                g.format_csv_device(stamp, hops.start, len(hops), p_db, g.db_count, p_smp,
                                    text_dev[k].data_ptr() + offs[r], caps[r], lens + 8 * r)
                for gi, name in enumerate(groups[1:], 1):
                    q = gi * world + r
                    at, cap, ln = text_dev[k].data_ptr() + offs[q], caps[q], lens + 8 * q
                    if name == "sk":
                        g.format_sk_csv_device(stamp, hops.start, len(hops), gather.slot_sk(k, r)[1], g.db_count, p_smp,
                                               at, cap, ln)
                        continue
                    x_db, x_fl, x_smp = gather.slot_excise(k, r)     # the folded samples are the count column
                    if name == "excise":
                        g.format_csv_device(stamp, hops.start, len(hops), x_db, g.db_count, x_smp, at, cap, ln)
                    else:
                        g.format_sk_csv_device(stamp, hops.start, len(hops), x_fl, g.db_count, x_smp, at, cap, ln)
        gather.release_copy(k, stream)
        with torch.cuda.stream(stream):
            text_host[k].copy_(text_dev[k], non_blocking=True)
        text_ready[k].record(stream)

    def print_pending():
        gather.wait(pending)
        if rank == 0:
            text_ready[pending].synchronize()
            buf = text_host[pending].numpy()
            lens = buf[lens_at:].view(np.int64)
            for q in range(len(caps)):
                if len(gather.ranges[q % world]):
                    if lens[q] < 0:
                        raise RuntimeError("sweep_main: a report value is outside the CSV formatter's domain")
                    outs[groups[q // world]].append(buf[offs[q]: offs[q] + lens[q]].tobytes().decode())

    for interval in range(args.intervals):
        k = interval & 1
        if g:
            if consumed[k] is not None:
                consumed[k].synchronize()
            if rng is None:
                synth_cube(pinned[k].ptr, mode, args.seed, args.param, tc, mine.start, len(mine),
                           interval * args.sweeps, args.sweeps, b)
                # --excise: chunks of K passes, a fold behind each (the last, shorter chunk's fold comes before
                # the report); without it one chunk
                for p0 in range(0, args.sweeps, chunk):
                    g.submit_batch(0, len(mine), min(chunk, args.sweeps - p0), pinned[k].ptr + p0 * len(mine) * b,
                                   len(mine) * b, b)
                    if excise:
                        g.excise_fold(k_low, k_high)
            else:
                # randomised hopping: every sweep visits this rank's hops in its own random order
                cube = pinned[k].view(np.uint8, (args.sweeps, len(mine), b))
                order = np.stack([rng.permutation(len(mine)) for _ in range(args.sweeps)]).astype(np.int32)
                for s_ in range(args.sweeps):
                    for j, lh in enumerate(order[s_]):
                        host.synth_generate(mode, ctypes.c_uint64(args.seed), args.param, tc, mine.start + int(lh),
                                            ctypes.c_uint64(interval * args.sweeps + s_), cube[s_, j].ctypes.data,
                                            ctypes.c_size_t(b))
                for p0 in range(0, args.sweeps, chunk):
                    g.submit_reads(order[p0: p0 + chunk].ravel(), pinned[k].ptr + p0 * len(mine) * b, b)
                    if excise:
                        g.excise_fold(k_low, k_high)
            gather.before_collect(k, stream)
            if excise:
                # a peek, in front of the collect's read-and-zero of S1, S2 and the excision state
                g.excised_report_device(*gather.excise_pointers(k))
            if sk:
                g.collect_sk_device(*gather.pointers(k), None,
                                    gather.sk_pointers(k)[1] if args.sk_out is not None else None)
            else:
                g.collect_device(*gather.pointers(k))
            consumed[k] = torch.cuda.Event()
            consumed[k].record(stream)
        # one exchange per interval (asynchronous, second stream); the previous interval's rows are
        # printed while this one is on the GPU
        gather.publish(k, stream)
        if rank == 0:
            format_rows(k)
        if pending is not None:
            print_pending()
        pending = k
    if pending is not None:
        print_pending()
    if rank == 0:
        _write_rows(args, outs["power"], outs.get("sk", []), outs.get("excise"), outs.get("flags"))
    if rank == 0:
        # torch's pinned-memory allocator records an event on the stream of the last copy when it frees a block:
        # the text buffers go before the handle's stream does
        stream.synchronize()
        text_host.clear()
    if g:
        g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _write_rows(args, rows_out, sk_rows_out, excise_rows=None, flag_rows=None):
    text = "".join(rows_out)
    if args.out == "-":
        sys.stdout.write(text)
    else:
        with open(args.out, "w") as f:
            f.write(text)
    for path, rows in ((args.sk_out, sk_rows_out), (args.excise_out, excise_rows), (args.flags_out, flag_rows)):
        if path is not None:
            with open(path, "w") as f:
                f.write("".join(rows))


def _main_read_sharded(args, rs, host, plan, pd, mode, world, rank, local, torch, dist,
                       SpectrumGather, shard_hops, synth_cube):
    """--shard reads: rank r transforms sweeps [S*r/W, S*(r+1)/W) of every interval for ALL hops; rank 0 merges"""
    tc, b, n = pd["tune_count"], pd["buf_len"], 1 << pd["bin_e"]
    sweeps = shard_hops(args.sweeps, world, rank)            # the same balanced split, over sweeps
    window = rs.window_coefs(args.window, n) if pd["bin_e"] else None
    sk = args.sk_out is not None
    g = rs.GpuScan.from_plan(pd, window_coefs=window, device=local, spectral_kurtosis=sk,
                             guard_bits=args.guard_bits)
    gather = SpectrumGather(tc, n, g.db_count, world, rank, torch.device("cuda", local),
                            mode=("host" if args.backend == "gloo" and world > 1 else None), replicated=True, sk=sk)
    if rank == 0 and world > 1:
        print("sweep_main: reads sharded %s over %d ranks; partial accumulators: %s" % (
            [len(shard_hops(args.sweeps, world, r)) for r in range(world)], world, gather.describe()), file=sys.stderr)
    stream = torch.cuda.ExternalStream(g.get_stream())
    if rank == 0:
        g.set_csv_columns(*plan.csv_columns())
    pinned = [rs.PinnedBuffer(max(1, len(sweeps) * tc * b)) for _ in range(2)]
    consumed = [None, None]
    rows_out, sk_rows_out = [], []
    for interval in range(args.intervals):
        k = interval & 1
        if consumed[k] is not None:
            consumed[k].synchronize()
        if len(sweeps):
            synth_cube(pinned[k].ptr, mode, args.seed, args.param, tc, 0, tc,
                       interval * args.sweeps + sweeps.start, len(sweeps), b)
            g.submit_batch(0, tc, len(sweeps), pinned[k].ptr, tc * b, b)
        gather.before_collect(k, stream)
        p_avg, p_smp, _ = gather.pointers(k)
        # raw sums + counts only: dB and SK come from the merged integers
        if sk:
            g.collect_sk_device(p_avg, p_smp, None, gather.sk_pointers(k)[0], None)
        else:
            g.collect_device(p_avg, p_smp, None)
        consumed[k] = torch.cuda.Event()
        consumed[k].record(stream)
        gather.publish(k, stream)
        if rank == 0:
            stream.wait_event(gather.gathered[k])
            if sk:
                s_avg, s_smp, sets, stride = gather.partial_sets(k)
                g.merge_sk_device(s_avg, s_smp, gather.sk_sections(s_avg)[0], sets, stride)
                text, sk_text = g.collect_sk_csv(args.stamp + ", ")
                rows_out.append(text.decode())
                sk_rows_out.append(sk_text.decode())
            else:
                g.merge_device(*gather.partial_sets(k))
                rows_out.append(g.collect_csv(args.stamp + ", ").decode())
    if rank == 0:
        _write_rows(args, rows_out, sk_rows_out)
    torch.cuda.synchronize()
    g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
