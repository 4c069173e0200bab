#!/usr/bin/env python
"""Per-kernel SASS opcode census of csrc/liblewin_b200.so (cuobjdump -sass): the mnemonics that prove which datapath a
kernel uses — UTCHMMA (tcgen05.mma), LDTM / STTM (tcgen05.ld / st), UTMALDG / UTMASTG (TMA load / store), UTCBAR
(tcgen05.commit), HMMA (mma.sync), LDSM (ldmatrix), LDGSTS (cp.async), SYNCS (mbarrier).  Runs without a GPU.

    python scripts/sass_census.py > profiles/r2_sass_census.txt
    python scripts/sass_census.py --compare OTHER.so      # per kernel: same instructions as in OTHER.so (e.g. a parent build)?

--compare matches kernels by demangled name, treating an added trailing `false` template argument (a new `bool` parameter
defaulting to the old code, such as the deterministic-mode DET switch) as the old name; it reports kernels whose instruction
text is identical, kernels that differ only in register numbering, kernels that differ otherwise, and new kernels.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "research-and-implementation-of-image-dehazing-algorithm-based-on-vision-transformer_b200", "csrc", "liblewin_b200.so")
OPS = ("UTCHMMA", "UTCQMMA", "LDTM", "STTM", "UTCBAR", "UTMALDG", "UTMASTG", "HMMA", "LDSM", "LDGSTS", "SYNCS", "MUFU", "FFMA2", "ATOMS", "RED")


def _instructions(lib):
    """{demangled kernel name: [instruction text]}"""
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    per, cur = collections.OrderedDict(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and cur:
            per[cur].append(m.group(1).strip())
    names = list(per)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return {re.sub(r"^void ", "", d): per[n] for n, d in zip(names, dem)}


def compare(other):
    old, new = _instructions(other), _instructions(LIB)
    cands = lambda d: (d, re.sub(r", false>\(", ">(", d), d.replace("<false>(", "("))
    regs = lambda ins: [re.sub(r"\bU?R\d+\b", "R", i) for i in ins]
    same, renamed, differ, added, seen = [], [], [], [], set()
    for d, ins in new.items():
        o = next((c for c in cands(d) if c in old), None)
        if o is None:
            added.append((d, len(ins)))
            continue
        seen.add(o)
        (same if old[o] == ins else renamed if regs(old[o]) == regs(ins) else differ).append(o)
    short = lambda d: re.sub(r"\(.*", "", d).replace("lewin::", "").replace("(anonymous namespace)::", "")
    print(f"# {len(old)} kernels in {os.path.basename(other)}: {len(same)} identical instruction for instruction, "
          f"{len(renamed)} identical up to register numbering, {len(differ)} different, {len(set(old) - seen)} absent here")
    for tag, lst in (("renumbered", renamed), ("DIFFERENT", differ)):
        for d in lst:
            print(f"{tag}: {short(d)}")
    for d in sorted(set(old) - seen):
        print(f"absent: {short(d)}")
    print(f"# {len(added)} new kernels")
    for d, n in added:
        print(f"new: {short(d)[:100]:100s} n={n}")
    return 1 if differ or set(old) - seen else 0


def main():
    if len(sys.argv) == 3 and sys.argv[1] == "--compare":
        return compare(sys.argv[2])
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    demangle = {}
    per = collections.OrderedDict()
    cur = None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur:
            per[cur][m.group(1)] += 1
            per[cur]["_total"] += 1
    names = list(per)
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    demangle = dict(zip(names, out))
    tot = collections.Counter()
    print("# SASS opcode census of liblewin_b200.so (sm_100a), one line per kernel: instructions, then the counts of the datapath mnemonics")
    print("# " + " ".join(OPS))
    for k in names:
        c = per[k]
        d = re.sub(r"\(.*", "", demangle.get(k, k))
        d = d.replace("void ", "").replace("lewin::", "").replace("(anonymous namespace)::", "")
        cols = " ".join(f"{op}={c[op]}" for op in OPS if c[op])
        print(f"{d[:110]:110s} n={c['_total']:6d}  {cols}")
        for op in OPS:
            tot[op] += c[op]
    print("# totals: " + " ".join(f"{op}={tot[op]}" for op in OPS))


if __name__ == "__main__":
    sys.exit(main())
