"""Instruction histogram per kernel of the built library (cuobjdump -sass): the Blackwell-native evidence SURVEY.md's last
paragraph names for this project -- sm_100a SASS with 128-bit LDG/STG, RED/ATOM on the histogram and the delta cells,
release/acquire at system scope and stores to peer-mapped memory in the sharded kernels (no tensor-core work exists on this
path).   python tools/sass_histogram.py [lib.so] > profiles/r02_sass_histogram.md"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "bpe_tokenizer_b200", "libbpe_b200.so")
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
arch = sorted(set(re.findall(r"arch = (sm_\w+)", out)))
kernels = collections.OrderedDict()
cur = None
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = m.group(1)
        d = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
        cur = re.sub(r"\(.*", "", d).replace("bpe::", "")
        kernels[cur] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)", line)
    if m and cur:
        kernels[cur][m.group(1)] += 1

INTEREST = [("128-bit global loads", r"^LDG\.E\.128"), ("128-bit global stores", r"^STG\.E\.128"), ("64-bit global loads", r"^LDG\.E\.64"),
            ("global atomics with return", r"^ATOMG"), ("global reductions (no return)", r"^REDG|^RED\."), ("shared atomics", r"^ATOMS"),
            ("system-scope strong ld/st", r"(LDG|STG|LD|ST).*\.STRONG\.SYS"), ("gpu-scope strong ld/st", r"(LDG|STG|LD|ST).*\.STRONG\.GPU"),
            ("MEMBAR", r"^MEMBAR"), ("L1 invalidate", r"^CCTL"), ("warp match/vote/shuffle", r"^MATCH|^VOTE|^SHFL|^REDUX"),
            ("packed u16x2 min/max", r"^VIMNMX.*U16x2|^VIMNMX.*U16X2"), ("prefetch", r"^CCTL.*PF|^LDG.*\.PF|^PREFETCH"), ("cp.async / bulk", r"^LDGSTS|^UBLKCP|^UTMA"),
            ("tensor core", r"^UTC|^HMMA|^HGMMA|^IMMA|^LDTM|^STTM")]
print("# SASS instruction histogram of libbpe_b200.so (%s; `cuobjdump -sass`, `tools/sass_histogram.py`)\n" % ", ".join(arch))
print("No kernel of this path is a contraction: no tensor-core, TMEM or TMA instruction appears (last row of every table stays 0);")
print("the Blackwell-relevant evidence is the memory instruction mix below.\n")
print("| kernel | instr | " + " | ".join(n for n, _ in INTEREST) + " |")
print("|---|---|" + "---|" * len(INTEREST))
for k, c in kernels.items():
    total = sum(c.values())
    if total < 40:
        continue
    row = []
    for _, pat in INTEREST:
        row.append(str(sum(v for op, v in c.items() if re.search(pat, op))))
    print("| `%s` | %d | %s |" % (k, total, " | ".join(row)))
print("\n## Full opcode lists of the hot kernels\n")
for k in ("k_merge_rounds", "k_merge_loop", "k_encode_lanes<20, 16>", "k_hist", "k_scatter"):
    for name, c in kernels.items():
        if name.startswith(k.split("<")[0]) and (k == name or "<" not in k):
            print("**`%s`**: " % name + ", ".join("%s x%d" % (op, v) for op, v in c.most_common(40)) + "\n")
            break
