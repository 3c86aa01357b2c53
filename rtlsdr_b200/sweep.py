"""Hop-sharded sweeps over the GPUs of one box.

Frequency hops are independent (reference src/rtl_power.c:650-719: tunes[i] are
disjoint), so hops are dealt to ranks in contiguous ranges and every rank runs
its own rtlsdr_gpu_scan handle; there is no collective on the data path.  Once
per integration interval the per-hop spectra (int64 bins, dB doubles, sample
counts) reach rank 0 with ONE exchange, and rank 0 prints the rows in hop order
like the reference's report loop (rtl_power.c:995-1000).

One process per GPU; torch.distributed is only the plumbing (NCCL over NVLink
on the GPU box, gloo in the CPU tests).

Three forms of the per-interval exchange, chosen once for all ranks:
  peer   every rank's report epilogue (rtlsdr_gpu_scan_collect_device) stores
         straight into its slot of rank 0's buffer through an NVLink peer mapping
         (torch symmetric memory).  No copy, no collective kernel: a one-thread
         kernel behind the epilogue raises the rank's "slot complete" flag in rank
         0's memory, rank 0 waits for all flags on a second stream with a kernel
         whose threads sleep between polls, (copies the report out,) and raises
         an "interval consumed" flag in every rank's memory, which a rank awaits
         before it rewrites that buffer two intervals later
         (rtlsdr_gpu_scan_flag_signal / _flag_wait).  A spinning barrier kernel or a
         collective's CTAs would take issue slots from the transform kernel on the
         SM they land on, and with its static equal-run schedule one slowed SM
         delays the whole launch (measured at 8 GPUs: 545 vs 513 us per interval).
  nccl   ONE torch.distributed.gather (grouped send/receive) per interval on a
         second stream (RTLSDR_B200_NCCL_GATHER=1, or no peer access).
  host   gloo / CPU tensors (tests; also CUDA ranks without NCCL: the report is
         staged through host memory).

Ordering rules this class owns (ADVICE r1): a rank never rewrites a report buffer
before the exchange that consumed it has finished (`before_collect`), and rank 0
copies a gathered report out before any rank may overwrite it (peer: the
"interval consumed" flag is raised behind that copy; nccl / host: the exchange of
interval j+1 is ordered behind the copy on rank 0's second stream, and every rank's
epilogue j+2 waits for exchange j+1).
"""
import os
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch
import torch.distributed as dist

SLOTS = 2  # report buffers: interval j+1 is transformed while interval j is exchanged


def shard_hops(tune_count: int, world: int, rank: int) -> range:
    """Contiguous, balanced hop range of `rank`: sizes differ by at most one."""
    base, extra = divmod(tune_count, world)
    lo = rank * base + min(rank, extra)
    return range(lo, lo + base + (1 if rank < extra else 0))


def max_hops_per_rank(tune_count: int, world: int) -> int:
    return -(-tune_count // world)


def shard_ranges(tune_count: int, world: int, sizes=None) -> List[range]:
    """Contiguous hop range of every rank: balanced (shard_hops) or with the given sizes (sum = tune_count),
    e.g. proportional to each GPU's measured host-to-device bandwidth for host-fed sweeps."""
    if sizes is None:
        return [shard_hops(tune_count, world, r) for r in range(world)]
    assert len(sizes) == world and sum(sizes) == tune_count and min(sizes) >= 0
    out, lo = [], 0
    for n in sizes:
        out.append(range(lo, lo + n))
        lo += n
    return out


def weighted_sizes(tune_count: int, weights) -> List[int]:
    """integer shares of tune_count proportional to `weights` (largest remainders), at least one hop per rank
    when there are enough hops"""
    w = [max(float(x), 0.0) for x in weights]
    total = sum(w) or 1.0
    exact = [tune_count * x / total for x in w]
    sizes = [int(e) for e in exact]
    if tune_count >= len(w):
        sizes = [max(1, n) for n in sizes]
    order = sorted(range(len(w)), key=lambda i: exact[i] - int(exact[i]), reverse=True)
    i = 0
    while sum(sizes) < tune_count:
        sizes[order[i % len(w)]] += 1
        i += 1
    order = sorted(range(len(w)), key=lambda i: sizes[i], reverse=True)
    i = 0
    while sum(sizes) > tune_count:
        j = order[i % len(w)]
        if sizes[j] > 1:
            sizes[j] -= 1
        i += 1
    return sizes


@dataclass
class IntervalReport:
    avg: np.ndarray       # [tune_count, N] int64, natural FFT order
    db: np.ndarray        # [tune_count, db_count] float64
    samples: np.ndarray   # [tune_count] int32
    s2: Optional[np.ndarray] = None   # sk: [tune_count, N, 2] uint64 (lo, hi) sums of |X|^4
    sk: Optional[np.ndarray] = None   # sk: [tune_count, db_count] float64 SK rows


class SpectrumGather:
    """One rank's side of the per-interval exchange.

    A report buffer is `words` int64 words: [avg hmax*N | db hmax*db_count (bit patterns) |
    samples hmax x int32, padded to 8 bytes], hmax = the largest shard; with sk=True (spectral-kurtosis handles)
    followed by [S2 hmax*N*2 (lo, hi) | SK rows hmax*db_count], at word offsets s2_at and sk_at.  Use per interval j
    (k = j % SLOTS):
        before_collect(k, stream); collect_device(*pointers(k)); publish(k, stream)
        (sk: collect_sk_device(*pointers(k), *sk_pointers(k)))
        ... later, rank 0: fetch(k)  (needs publish(..., to_host=True))
    """

    def __init__(self, tune_count, n_bins, db_count, world, rank, device, mode=None, sizes=None, replicated=False,
                 sk=False):
        self.tune_count, self.n, self.db_count = tune_count, n_bins, db_count
        self.world, self.rank = world, rank
        self.device = torch.device(device)
        self.cuda = self.device.type == "cuda"
        # replicated: every rank reports ALL hops (the reads of the hops are sharded instead, see ReadShardedMerge);
        # rank 0 then holds `world` partial accumulator sets per interval instead of disjoint hop ranges
        self.replicated = replicated
        self.ranges = [range(tune_count)] * world if replicated else shard_ranges(tune_count, world, sizes)
        self.hmax = max(1, max(len(r) for r in self.ranges))
        self.smp_words = (self.hmax + 1) // 2
        self.words = self.hmax * (n_bins + db_count) + self.smp_words
        self.sk = sk
        self.s2_at = self.sk_at = None
        if sk:
            self.s2_at = self.words
            self.sk_at = self.s2_at + self.hmax * n_bins * 2
            self.words = self.sk_at + self.hmax * db_count
        self.my_hops = self.ranges[rank]
        self.peer = None
        # peer mode: int32 flags behind the report buffers of the symmetric allocation:
        # [SLOTS][world] "slot complete" (used in rank 0's copy), [SLOTS] "interval consumed" (every rank's own copy), [1] time-out
        self.flag_words = (SLOTS * world + SLOTS + 2 + 1) // 2
        self.seq = [0] * SLOTS
        if mode is None:
            mode = self._pick_mode()
        if mode == "peer" and not self._setup_peer():
            mode = "nccl"
        self.mode = mode
        self.last_exchange = None
        if self.cuda:
            self.comm = torch.cuda.Stream(device=self.device)
            self.ready = [torch.cuda.Event() for _ in range(SLOTS)]
            self.gathered = [torch.cuda.Event() for _ in range(SLOTS)]
        if mode == "peer":
            buf = self.peer[0]
            self.send = [buf[(k * world + rank) * self.words:(k * world + rank + 1) * self.words] for k in range(SLOTS)]
            self.recv = ([buf[k * world * self.words:(k + 1) * world * self.words].view(world, self.words)
                          for k in range(SLOTS)] if rank == 0 else None)
        else:
            dev = self.device
            self.send = [torch.zeros(self.words, dtype=torch.int64, device=dev) for _ in range(SLOTS)]
            rdev = torch.device("cpu") if mode == "host" else dev
            self.recv = ([torch.zeros(world, self.words, dtype=torch.int64, device=rdev) for _ in range(SLOTS)]
                         if rank == 0 else None)
        if mode == "host" and self.cuda:
            self.stage = [torch.zeros(self.words, dtype=torch.int64).pin_memory() for _ in range(SLOTS)]
        # rank 0, replicated: private device copy of a gathered buffer, made before the writers may reuse the slots
        self.dev_copy = None
        self.copy_free = [None] * SLOTS     # events after which dev_copy[k] may be overwritten (release_copy)
        if replicated and rank == 0 and self.cuda:
            self.dev_copy = [torch.zeros(world, self.words, dtype=torch.int64, device=self.device) for _ in range(SLOTS)]
        # rank 0: pinned landing area of a gathered report
        self.host = None
        if rank == 0 and self.cuda and mode != "host":
            self.host = [torch.zeros(world, self.words, dtype=torch.int64).pin_memory() for _ in range(SLOTS)]

    # ---- setup ----------------------------------------------------------------

    def _pick_mode(self):
        if self.world == 1:
            return "nccl" if self.cuda else "host"   # no exchange; "nccl" = device buffers
        if not self.cuda or dist.get_backend() != "nccl":
            return "host"
        return "nccl" if os.environ.get("RTLSDR_B200_NCCL_GATHER") else "peer"

    def _agree(self, ok):
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return int(flag.item()) == 1

    def _setup_peer(self):
        """Symmetric-memory buffer on every rank (rank 0's is the destination).  The rendezvous is a
        collective, so the ranks first agree that everybody can reach it (import + allocation), and
        agree again on its outcome; any failure anywhere -> every rank takes the NCCL gather."""
        symm = buf = None
        try:
            import torch.distributed._symmetric_memory as symm
            # only rank 0's copy is ever written, but the allocation is symmetric by construction
            buf = symm.empty(SLOTS * self.world * self.words + self.flag_words, dtype=torch.int64, device=self.device)
            buf.zero_()
            torch.cuda.synchronize(self.device)   # flags are zero before any peer can raise one
            ok = True
        except Exception:  # noqa: BLE001
            ok = False
        if not self._agree(ok):
            return False
        hdl = None
        try:
            hdl = symm.rendezvous(buf, dist.group.WORLD)
            root = int(hdl.buffer_ptrs[0])
            self.peer_ptrs = [int(p) for p in hdl.buffer_ptrs]
            ok = True
        except Exception:  # noqa: BLE001
            ok = False
        if not self._agree(ok):
            return False
        self.peer = (buf, hdl, root)
        return True

    # ---- per interval -----------------------------------------------------------

    def pointers(self, k=0):
        """device addresses for rtlsdr_gpu_scan_collect_device(avg, samples(int32), db) of report buffer k:
        this rank's slot of rank 0's buffer in peer mode, the local send buffer otherwise"""
        if self.mode == "peer":
            base = self.peer[2] + (k * self.world + self.rank) * self.words * 8
        else:
            base = self.send[k].data_ptr()
        p_db = base + self.hmax * self.n * 8
        p_smp = p_db + self.hmax * self.db_count * 8
        return base, p_smp, p_db

    def sk_pointers(self, k=0):
        """sk: device addresses of S2 and the SK rows for rtlsdr_gpu_scan_collect_sk_device() of report buffer k,
        behind pointers(k)'s sections of the same slot"""
        return self.sk_sections(self.pointers(k)[0])

    def sk_sections(self, slot_base):
        """sk: (address of S2, address of the SK rows) of the slot starting at `slot_base`; slots are words * 8
        bytes apart, so merge_sk_device() walks the S2 of consecutive slots with that stride"""
        assert self.sk
        return slot_base + self.s2_at * 8, slot_base + self.sk_at * 8

    def views(self, k=0):
        """(avg [h, N] int64, db [h, db_count] float64, samples [h] int32) views of the LOCAL send buffer k
        sized for this rank's hop count (host mode / tests fill these instead of a GPU epilogue); with sk also
        (s2 [h, N, 2] uint64, sk [h, db_count] float64)"""
        h = len(self.my_hops)
        s = self.send[k]
        a = s[: self.hmax * self.n].view(self.hmax, self.n)[:h]
        o = self.hmax * self.n
        d = s[o: o + self.hmax * self.db_count].view(torch.float64).view(self.hmax, self.db_count)[:h]
        o += self.hmax * self.db_count
        c = s[o: o + self.smp_words].view(torch.int32)[:h]
        if not self.sk:
            return a, d, c
        s2 = s[self.s2_at: self.sk_at].view(torch.uint64).view(self.hmax, self.n, 2)[:h]
        sk = s[self.sk_at: self.words].view(torch.float64).view(self.hmax, self.db_count)[:h]
        return a, d, c, s2, sk

    def _flag_addr(self, owner, index):
        """device address (as seen from this rank) of int32 flag `index` in rank `owner`'s symmetric buffer"""
        return self.peer_ptrs[owner] + SLOTS * self.world * self.words * 8 + 4 * index

    def before_collect(self, k, stream=None):
        """Call before the epilogue writes report buffer k (on the stream the epilogue will run on).
        peer: that stream waits until rank 0 has consumed the buffer's previous content (its "interval consumed"
        flag, raised behind rank 0's copy-out).  Otherwise: it waits for the most recent exchange (which, on rank
        0, is ordered behind the copy-out of the exchange before it)."""
        if not self.cuda or self.world == 1:
            return
        stream = stream or torch.cuda.current_stream()
        if self.mode == "peer":
            if self.seq[k] > 0:
                from .scan import flag_wait
                flag_wait(stream.cuda_stream, self._flag_addr(self.rank, SLOTS * self.world + k), 1, self.seq[k],
                          0, self._flag_addr(self.rank, SLOTS * self.world + SLOTS))
        elif self.last_exchange is not None:
            stream.wait_event(self.last_exchange)

    def publish(self, k, stream=None, to_host=False):
        """Report buffer k is complete once everything enqueued so far on `stream` has run: exchange it on the
        second stream (asynchronous on CUDA).  to_host: rank 0 also copies the gathered report to pinned memory."""
        if not self.cuda:
            if self.world > 1:
                dist.gather(self.send[k], list(self.recv[k].unbind(0)) if self.rank == 0 else None, dst=0)
            elif self.rank == 0:
                self.recv[k][0].copy_(self.send[k])
            return
        stream = stream or torch.cuda.current_stream()
        if self.mode == "peer" and self.world > 1:
            from .scan import flag_signal, flag_signal_many, flag_wait
            self.seq[k] += 1
            seq = self.seq[k]
            # "my slot of buffer k is complete": into rank 0's memory, behind this rank's epilogue
            flag_signal(stream.cuda_stream, self._flag_addr(0, k * self.world + self.rank), seq)
            if self.rank != 0:
                self.gathered[k].record(stream)
                self.last_exchange = self.gathered[k]
                return
            with torch.cuda.stream(self.comm):
                flag_wait(self.comm.cuda_stream, self._flag_addr(0, k * self.world), self.world, seq, 0,
                          self._flag_addr(0, SLOTS * self.world + SLOTS))
                if to_host:
                    self.host[k].copy_(self.recv[k], non_blocking=True)
                if self.dev_copy is not None:
                    if self.copy_free[k] is not None:
                        self.comm.wait_event(self.copy_free[k])
                    self.dev_copy[k].copy_(self.recv[k], non_blocking=True)
                # "interval consumed" in every rank's memory (one launch): the slots may be rewritten
                addrs = [self._flag_addr(r, SLOTS * self.world + k) for r in range(self.world)]
                for lo in range(0, self.world, 32):
                    flag_signal_many(self.comm.cuda_stream, addrs[lo:lo + 32], seq)
                self.gathered[k].record(self.comm)
            self.last_exchange = self.gathered[k]
            return
        self.ready[k].record(stream)
        with torch.cuda.stream(self.comm):
            self.comm.wait_event(self.ready[k])
            if self.world == 1:
                src = self.send[k].view(1, self.words)
            elif self.mode == "nccl":
                dist.gather(self.send[k], list(self.recv[k].unbind(0)) if self.rank == 0 else None, dst=0)
                src = self.recv[k] if self.rank == 0 else None
            else:  # host staged (gloo with CUDA ranks)
                self.stage[k].copy_(self.send[k], non_blocking=True)
                self.comm.synchronize()
                dist.gather(self.stage[k], list(self.recv[k].unbind(0)) if self.rank == 0 else None, dst=0)
                src = None
            if to_host and self.rank == 0 and src is not None:
                self.host[k].copy_(src, non_blocking=True)
            if self.dev_copy is not None:
                if self.copy_free[k] is not None:
                    self.comm.wait_event(self.copy_free[k])
                self.dev_copy[k].copy_(src if src is not None else self.recv[k], non_blocking=True)
            self.gathered[k].record(self.comm)
        self.last_exchange = self.gathered[k]

    def drain(self, stream=None):
        """make `stream` wait for every exchange issued so far"""
        if self.cuda:
            (stream or torch.cuda.current_stream()).wait_stream(self.comm)

    def fetch(self, k) -> Optional[IntervalReport]:
        """rank 0: the gathered report of buffer k (blocks until its exchange and copy-out are done)"""
        if self.cuda:
            self.gathered[k].synchronize()
        if self.rank != 0:
            return None
        if self.mode == "peer" and self.world > 1:
            flags = self.peer[0][SLOTS * self.world * self.words:].view(torch.int32)
            if int(flags[SLOTS * self.world + SLOTS].item()) != 0:
                raise RuntimeError("SpectrumGather: a rank's report did not arrive within the flag wait's time-out")
        if self.mode == "host" or not self.cuda:
            bufs = self.recv[k].numpy()
        else:
            bufs = self.host[k].numpy()
        return self.unpack(bufs)

    def wait(self, k):
        """block until the exchange of buffer k is done; raises if a rank's report did not arrive (peer mode)"""
        if self.cuda:
            self.gathered[k].synchronize()
        if self.rank == 0 and self.mode == "peer" and self.world > 1:
            flags = self.peer[0][SLOTS * self.world * self.words:].view(torch.int32)
            if int(flags[SLOTS * self.world + SLOTS].item()) != 0:
                raise RuntimeError("SpectrumGather: a rank's report did not arrive within the flag wait's time-out")

    def partial_sets(self, k):
        """rank 0, replicated mode: (device address of set 0's raw bins, of its int32 counts, number of sets, bytes
        between sets) of the gathered buffer k, for rtlsdr_gpu_scan_merge_device() on a stream that has waited for
        `gathered[k]`.  The copy was made before any rank may rewrite its slot."""
        assert self.replicated and self.rank == 0 and self.dev_copy is not None
        base = self.dev_copy[k].data_ptr()
        smp = base + (self.hmax * self.n + self.hmax * self.db_count) * 8
        return base, smp, self.world, self.words * 8

    def keep_device_copy(self):
        """rank 0, CUDA: from now on every exchange also leaves a private device copy of the gathered buffer (made
        on the second stream before any rank may rewrite its slot; from the host buffer in host mode), for readers
        on another stream such as the CSV formatter.  They call release_copy() behind their last read."""
        if self.rank == 0 and self.cuda and self.dev_copy is None:
            self.dev_copy = [torch.zeros(self.world, self.words, dtype=torch.int64, device=self.device)
                             for _ in range(SLOTS)]

    def slot_rows(self, k, r):
        """rank 0: (device address of the dB rows, of the int32 counts) of rank r's slot in the private copy of
        buffer k (keep_device_copy); the dB rows are db_count doubles apart"""
        base = self.dev_copy[k].data_ptr() + r * self.words * 8
        p_db = base + self.hmax * self.n * 8
        return p_db, p_db + self.hmax * self.db_count * 8

    def slot_sk(self, k, r):
        """rank 0, sk: (device address of S2, of the SK rows) of rank r's slot in the private copy of buffer k"""
        return self.sk_sections(self.dev_copy[k].data_ptr() + r * self.words * 8)

    def release_copy(self, k, stream):
        """rank 0, replicated mode: everything enqueued so far on `stream` (the merge) is the last reader of the
        private copy of buffer k; the exchange two intervals later waits for it before overwriting the copy"""
        ev = torch.cuda.Event()
        ev.record(stream)
        self.copy_free[k] = ev

    def unpack(self, bufs) -> IntervalReport:
        """bufs: int64 [world, words] -> rows in hop order"""
        avg = np.zeros((self.tune_count, self.n), dtype=np.int64)
        db = np.zeros((self.tune_count, self.db_count), dtype=np.float64)
        smp = np.zeros(self.tune_count, dtype=np.int32)
        s2 = np.zeros((self.tune_count, self.n, 2), dtype=np.uint64) if self.sk else None
        sk = np.zeros((self.tune_count, self.db_count), dtype=np.float64) if self.sk else None
        for r in range(self.world):
            hops = self.ranges[r]
            h = len(hops)
            if h == 0:
                continue
            b = bufs[r]
            avg[hops.start: hops.stop] = b[: self.hmax * self.n].reshape(self.hmax, self.n)[:h]
            o = self.hmax * self.n
            db[hops.start: hops.stop] = b[o: o + self.hmax * self.db_count].view(np.float64).reshape(
                self.hmax, self.db_count)[:h]
            o += self.hmax * self.db_count
            smp[hops.start: hops.stop] = b[o: o + self.smp_words].view(np.int32)[:h]
            if self.sk:
                s2[hops.start: hops.stop] = b[self.s2_at: self.sk_at].view(np.uint64).reshape(self.hmax, self.n, 2)[:h]
                sk[hops.start: hops.stop] = b[self.sk_at: self.words].view(np.float64).reshape(
                    self.hmax, self.db_count)[:h]
        return IntervalReport(avg, db, smp, s2, sk)

    def describe(self):
        return {"peer": "every rank's report epilogue stores its int64 bins + dB + counts straight into rank 0's "
                        "buffer over NVLink (symmetric-memory peer mapping); per interval one 'slot complete' flag per "
                        "rank and one 'consumed' flag back, raised by one-thread kernels and awaited by a sleeping "
                        "kernel on a second stream (no collective, no spinning CTA beside the transform)",
                "nccl": "one NCCL gather of int64 bins + dB + counts per interval, on a second stream, overlapped "
                        "with the next interval's transform",
                "host": "reports staged through host memory and gathered with torch.distributed (gloo)"}[self.mode] \
            if self.world > 1 else "none (one rank)"
