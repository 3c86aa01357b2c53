"""Per-kernel SASS signature of a built library: instruction count, hash of the SASS text, hash of the sorted
opcode list.  Two builds whose kernels have the same signatures run the same instructions.

    python tools/sass_sig.py LIB.so [--norm-regs] [--norm-params]

--norm-regs masks register numbers (R, UR, P, UP); --norm-params masks kernel-parameter offsets c[0x0][...]."""
import collections
import hashlib
import re
import subprocess
import sys


def sig(lines):
    return hashlib.sha1("\n".join(lines).encode()).hexdigest()[:12]


out = subprocess.run(["cuobjdump", "-sass", sys.argv[1]], capture_output=True, text=True, check=True).stdout
funcs, cur = collections.OrderedDict(), None
for line in out.splitlines():
    m = re.match(r"\s+Function : (\S+)", line)
    if m:
        cur = m.group(1)
        funcs[cur] = []
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(.*?);", line)
    if cur and m:
        txt = re.sub(r"\s+", " ", m.group(1))
        if "--norm-regs" in sys.argv:
            txt = re.sub(r"\bU?[RP]\d+\b", "R", txt)
        if "--norm-params" in sys.argv:
            txt = re.sub(r"c\[0x0\]\[[^]]*\]", "c[0x0][]", txt)
        funcs[cur].append(txt)
for f, ins in funcs.items():
    ops = sorted(re.sub(r"^@!?U?P\w+ ", "", i).split(" ")[0] for i in ins)
    print(sig(ins), sig(ops), len(ins), f)
