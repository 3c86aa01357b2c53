#!/usr/bin/env python
"""Instruction budget of a transform kernel's loops, counted on the CPU from the SASS.

    python tools/sass_budget.py [--lib LIB.so | --cubin X.cubin [--src TREE]] --kernel 'scan_small_kernel<12,0,0>'
                                [--kernel ...] [--max-ws N] [--max-alu N] [--lines K]

Without --lib / --cubin the library is built into a temporary directory with the flags of rtlsdr_b200/_build.py
(which include -lineinfo).  The SASS is disassembled with `nvdisasm -gi`, so every instruction carries the chain of
source lines it was inlined through.  Those lines are read from --src, the tree a given --lib / --cubin was built
from (default: this repository); the tool stops if a source file there is missing or newer than the binary.

The working-set loop is the innermost loop (back edge of a branch) that holds the transpose code (exchange /
exchange_pk); the per-read loop is the innermost loop around it.  For the working-set loop the tool prints the
instructions per thread by pipe and by bucket, with the source lines that issue the most of them; for the read
loop it prints the part outside the working-set loop: the head (from the read loop's start to the working-set loop)
runs once per read, the tail holds the rarely taken hop flush.

Pipes: FMA-heavy = IMAD*, IDP*; LSU = shared / global / constant memory, shuffles, atomics; other = barriers,
branches, uniform-datapath ops and other control; ALU = the rest (shifts, LOP3, LEA, PRMT, IADD3, compares ...).
--max-ws / --max-alu make the tool exit with status 1 when the working-set loop (of every kernel given) is longer,
or has more ALU-pipe instructions, than the budget."""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rtlsdr_b200", "csrc")

# function name -> bucket; the innermost frame of an instruction's inline chain that lies in one of these decides
BUCKET_OF_FUNC = {
    "butterfly": "butterflies", "butterfly_x": "butterflies", "butterfly_x_packed_b": "butterflies",
    "butterfly_x_re": "butterflies", "butterfly_x_im": "butterflies", "c16_re_fast": "butterflies",
    "run_pass": "butterflies",
    "exchange": "transposes", "exchange_pk": "transposes", "x_pack": "transposes", "x_unpack": "transposes",
    "xch_idx": "transposes",
    "accumulate_power": "|X|^2", "accumulate_power_sk": "|X|^2", "sk_accumulate": "|X|^2",
    "front_u8": "front end", "front_index": "front end",
    "get": "twiddle loads",
    "u8_read_dc": "DC sums",
    "cp_async16": "cp.async", "cp_async_commit": "cp.async", "cp_async_wait_all": "cp.async",
}
# lines of a textual kernel body (.inl) that are not inside a function: classified by what the line calls
BUCKET_OF_CALL = [("accumulate_power", "|X|^2"), ("front_u8", "front end"), ("cp_async", "cp.async"),
                  ("u8_read_dc", "DC sums")]
BUCKETS = ["butterflies", "transposes", "|X|^2", "front end", "twiddle loads", "DC sums", "cp.async", "other"]
PIPES = ["FMA", "ALU", "LSU", "other"]

LSU_OPS = ("LD", "ST", "LDS", "STS", "LDC", "LDG", "STG", "LDGSTS", "ATOM", "ATOMS", "ATOMG", "RED", "REDG",
           "SHFL", "LDSM", "LDGDEPBAR", "DEPBAR", "MEMBAR")


def pipe_of(op):
    base = op.split(".")[0]
    if base in ("IMAD", "IDP", "IMUL", "FFMA", "FMUL", "FADD", "FFMA2", "FMUL2", "FADD2", "HFMA2"):
        return "FMA"
    if base in LSU_OPS:
        return "LSU"
    if base in ("BAR", "BRA", "BSSY", "BSYNC", "EXIT", "RET", "CALL", "NOP", "WARPSYNC", "YIELD", "NANOSLEEP",
                "S2R", "S2UR", "CS2R", "ELECT", "VOTEU", "ACQBULK") or base.startswith("U") or base == "LDCU":
        return "other"
    return "ALU"


class Source:
    """function line ranges of the CUDA sources, for attributing inlined frames.

    A line-info path under rtlsdr_b200/csrc/ is read from the same place in `root`, the tree the binary was built
    from.  With `built` (the binary's modification time) a source file that is missing there or newer than the
    binary is an error: its line numbers would be attributed to code the binary was not built from."""

    def __init__(self, root, built=None):
        self.root, self.built = root, built
        self.funcs = {}   # path -> list of (first, last, name)
        self.text = {}

    def resolve(self, path):
        key = "rtlsdr_b200/csrc/"
        if key not in path:
            return path   # CUDA's own headers: no function of a bucket lives there
        real = os.path.join(self.root, key + path.split(key, 1)[1])
        if self.built is not None:
            if not os.path.exists(real):
                raise SystemExit(f"{real}: not found; pass --src with the tree the binary was built from")
            if os.path.getmtime(real) > self.built:
                raise SystemExit(f"{real} is newer than the binary; pass --src with the tree it was built from")
        return real

    def _load(self, path):
        if path in self.text:
            return
        try:
            with open(self.resolve(path)) as f:
                lines = f.read().split("\n")
        except OSError:
            lines = []
        self.text[path] = lines
        spans = []
        for i, ln in enumerate(lines):
            m = re.match(r"^(\s*)(?:template\s*<[^>]*>\s*)?SCAN_DEV\b[^;]*?\b(\w+)\s*\(", ln)
            if not m or ln.rstrip().endswith(";"):
                continue
            close = m.group(1) + "}"
            for j in range(i + 1, len(lines)):
                if lines[j].rstrip() == close:
                    spans.append((i + 1, j + 1, m.group(2)))
                    break
        self.funcs[path] = spans

    def func(self, path, line):
        self._load(path)
        best = None
        for a, b, name in self.funcs[path]:
            if a <= line <= b and (best is None or a > best[0]):
                best = (a, name)
        return best[1] if best else None

    def line(self, path, line):
        self._load(path)
        lines = self.text[path]
        return lines[line - 1] if 0 < line <= len(lines) else ""

    def bucket(self, chain):
        for path, line in chain:
            name = self.func(path, line)
            if name in BUCKET_OF_FUNC:
                return BUCKET_OF_FUNC[name]
            if name is None:
                txt = self.line(path, line)
                for key, b in BUCKET_OF_CALL:
                    if key in txt:
                        return b
        return "other"


def build_lib(tmp):
    sys.path.insert(0, ROOT)
    from rtlsdr_b200 import _build
    lib = os.path.join(tmp, "lib.so")
    subprocess.run([_build._nvcc()] + _build.NVCC_FLAGS + ["-o", lib, os.path.join(CSRC, "scan_abi.cu")], check=True)
    return lib


def cubins_of(lib, tmp):
    if lib.endswith(".cubin"):
        return [lib]
    d = os.path.join(tmp, "elf")
    os.makedirs(d, exist_ok=True)
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=d, check=True, capture_output=True)
    return sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith(".cubin"))


def norm_name(demangled):
    s = re.sub(r"\((?:int|bool|unsigned int)\)", "", demangled)  # cu++filt writes template arguments as (int)12
    s = re.sub(r"^void\s+", "", s.split("(")[0]).replace("rscan::", "").replace(" ", "")
    return s.replace("false", "0").replace("true", "1")


def disassemble(cubins):
    """mangled kernel name -> list of text lines of its section"""
    funcs = collections.OrderedDict()
    for cb in cubins:
        out = subprocess.run(["nvdisasm", "-gi", "-c", cb], capture_output=True, text=True, check=True).stdout
        cur = None
        for ln in out.split("\n"):
            m = re.match(r"//-+ \.text\.(\S+) -+", ln)
            if m:
                cur = m.group(1)
                funcs[cur] = []
            elif cur:
                funcs[cur].append(ln)
    return funcs


def demangle(names):
    out = subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.strip().split("\n")))


INS = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
LINE = re.compile(r'^\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')


def parse(lines):
    """-> instructions [(addr, text, opcode, chain)], labels {name: addr}"""
    ins, labels, chain, pending = [], {}, [], []
    for ln in lines:
        m = LINE.match(ln)
        if m:  # innermost frame first
            pending.append((m.group(1), int(m.group(2))))
            continue
        m = re.match(r"^(\.L_x_\d+):", ln)
        if m:
            labels[m.group(1)] = len(ins)
            continue
        m = INS.match(ln)
        if m:
            if pending:
                chain, pending = pending, []
            txt = re.sub(r"\s+", " ", m.group(2))
            body = re.sub(r"^@!?U?P\w+ ", "", txt)
            ins.append((int(m.group(1), 16), txt, body.split(" ")[0], chain))
    return ins, labels


def loops(ins, labels):
    """(first, last) instruction index of every loop: a branch back to a label at or before it"""
    out = []
    for i, (_, txt, op, _) in enumerate(ins):
        if op.startswith("BRA"):
            m = re.search(r"`\((\.L_x_\d+)\)", txt)
            if m and labels.get(m.group(1), i + 1) <= i:
                out.append((labels[m.group(1)], i))
    return out


def summarize(idx, ins, src):
    by_pipe, by_bucket, by_op, by_line = (collections.Counter() for _ in range(4))
    cross = collections.Counter()
    for i in idx:
        _, _, op, chain = ins[i]
        p, b = pipe_of(op), src.bucket(chain)
        by_pipe[p] += 1
        by_bucket[b] += 1
        by_op[op] += 1
        cross[b, p] += 1
        if chain:
            path, line = chain[0]
            by_line[os.path.basename(path), line, op] += 1
    return dict(n=len(idx), pipe=by_pipe, bucket=by_bucket, op=by_op, line=by_line, cross=cross)


def report(title, s, nlines):
    print(f"== {title}: {s['n']} instructions per thread")
    print("   " + "   ".join(f"{p} {s['pipe'][p]}" for p in PIPES))
    print(f"   {'bucket':14s} {'total':>6s} " + " ".join(f"{p:>6s}" for p in PIPES))
    for b in BUCKETS:
        if s["bucket"][b]:
            print(f"   {b:14s} {s['bucket'][b]:6d} " + " ".join(f"{s['cross'][b, p]:6d}" for p in PIPES))
    print("   opcodes: " + ", ".join(f"{op} {n}" for op, n in s["op"].most_common()))
    if nlines:
        print(f"   top source lines (innermost frame, opcode):")
        for (f, line, op), n in s["line"].most_common(nlines):
            print(f"     {n:5d}  {f}:{line}  {op}")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib")
    ap.add_argument("--cubin")
    ap.add_argument("--src", help="tree the --lib / --cubin was built from (default: this repository)")
    ap.add_argument("--kernel", action="append", required=True,
                    help="demangled name without spaces, bools as 0/1, e.g. 'scan_small_kernel<12,0,0>'")
    ap.add_argument("--max-ws", type=int)
    ap.add_argument("--max-alu", type=int)
    ap.add_argument("--lines", type=int, default=0, help="print the K source lines that issue the most instructions")
    a = ap.parse_args()

    fail = False
    with tempfile.TemporaryDirectory() as tmp:
        lib = a.cubin or a.lib or build_lib(tmp)
        src = Source(os.path.abspath(a.src or ROOT), None if lib.startswith(tmp) else os.path.getmtime(lib))
        funcs = disassemble(cubins_of(lib, tmp))
    names = demangle(list(funcs))
    for q in a.kernel:
        want = q.replace(" ", "")
        hits = [k for k in funcs if norm_name(names[k]) == want]
        if len(hits) != 1:
            print(f"{q}: {len(hits)} kernels match", file=sys.stderr)
            return 2
        ins, labels = parse(funcs[hits[0]])
        lps = loops(ins, labels)
        xch = {i for i, x in enumerate(ins) if src.bucket(x[3]) == "transposes"}
        cand = [(b - a_ + 1, a_, b) for a_, b in lps if any(a_ <= i <= b for i in xch)]
        if not cand:
            print(f"{q}: no loop holds the transposes", file=sys.stderr)
            return 2
        _, w0, w1 = min(cand)
        print(f"#### {q}  ({hits[0]}), {len(ins)} instructions")
        ws = summarize(range(w0, w1 + 1), ins, src)
        report(f"working-set loop {ins[w0][0]:#06x}..{ins[w1][0]:#06x}", ws, a.lines)
        outer = [(b - a_ + 1, a_, b) for a_, b in lps if a_ <= w0 and w1 <= b and (a_, b) != (w0, w1)]
        if outer:
            _, r0, r1 = min(outer)
            head = summarize(range(r0, w0), ins, src)
            tail = summarize(range(w1 + 1, r1 + 1), ins, src)
            report(f"read loop head {ins[r0][0]:#06x}..{ins[w0][0]:#06x} (once per read)", head, a.lines)
            report(f"read loop tail {ins[w1][0]:#06x}..{ins[r1][0]:#06x} (hop flush, mostly skipped)", tail, 0)
            print(f"== working set + half a read head (two working sets per read): {ws['n'] + head['n'] / 2:.1f}"
                  f"   ALU {ws['pipe']['ALU'] + head['pipe']['ALU'] / 2:.1f}")
        if a.max_ws is not None and ws["n"] > a.max_ws:
            print(f"{q}: working-set loop {ws['n']} > budget {a.max_ws}", file=sys.stderr)
            fail = True
        if a.max_alu is not None and ws["pipe"]["ALU"] > a.max_alu:
            print(f"{q}: working-set loop ALU pipe {ws['pipe']['ALU']} > budget {a.max_alu}", file=sys.stderr)
            fail = True
        print()
    return 1 if fail else 0


if __name__ == "__main__":
    sys.exit(main())
