"""Static view of every kernel in the shipped library (no GPU needed): per-kernel SASS instruction counts, registers,
local (spill) bytes, static shared memory, and the mnemonics that prove which hardware paths the code uses --
DMMA (FP64 tensor pipe), UBLKCP (1-D bulk TMA), SYNCS (mbarrier), UCGABAR / CGABAR (cluster barrier), MUFU, BAR.

    python tools/sass_summary.py [path/to/libapgp.so] > profiles/rNN_sass_summary.txt
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLS = ("DMMA", "UBLKCP", "SYNCS", "BAR", "DFMA", "DMUL", "DADD", "LDS", "STS", "MUFU", "CGABAR", "ATOM", "RED")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return dict(zip(names, out))


def short(name):
    name = re.sub(r"\(anonymous namespace\)::", "", name)
    name = re.sub(r"^void ", "", name)
    name = re.sub(r"apgp::", "", name)
    depth, cut = 0, len(name)
    for i, c in enumerate(name):                 # drop the argument list, keep template arguments
        if c == "<":
            depth += 1
        elif c == ">":
            depth -= 1
        elif c == "(" and depth == 0:
            cut = i
            break
    return name[:cut]


def collect(so):
    """[{kernel, instr, regs, local, smem, DMMA, UBLKCP, ...}] for every kernel in the shared library."""
    res = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True, check=True).stdout
    usage = {}
    fn = None
    for line in res.split("\n"):
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+).*?SHARED:(\d+).*?LOCAL:(\d+)", line)
        if m and fn:
            usage[fn] = (int(m.group(1)), int(m.group(3)), int(m.group(2)))
            fn = None
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    counts = collections.OrderedDict()
    cur = None
    for line in sass.split("\n"):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", line)
        if m and cur:
            op = m.group(1)
            counts[cur]["instr"] += 1
            if op.startswith("CGABAR") or op.startswith("UCGABAR"):
                counts[cur]["CGABAR"] += 1
            elif op in ("ATOM", "ATOMG", "ATOMS"):
                counts[cur]["ATOM"] += 1
            elif op in COLS:
                counts[cur][op] += 1
    names = demangle(list(counts))
    rows = []
    for fn, c in sorted(counts.items(), key=lambda kv: -kv[1]["instr"]):
        r = usage.get(fn, (0, 0, 0))
        row = {"kernel": short(names[fn]), "instr": c["instr"], "regs": r[0], "local": r[1], "smem": r[2]}
        row.update({k: c[k] for k in COLS})
        rows.append(row)
    return rows


def main():
    so = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "approxposterior_b200", "libapgp.so")
    print("cuobjdump -sass / -res-usage %s (sm_100a, built by __graft_entry__.build()); static instruction counts per kernel"
          % os.path.relpath(so, ROOT))
    print("%-64s %6s %5s %5s %8s " % ("kernel", "instr", "regs", "local", "smem(st)") + " ".join("%6s" % c for c in COLS))
    for r in collect(so):
        print("%-64s %6d %5d %5d %8d " % (r["kernel"][:64], r["instr"], r["regs"], r["local"], r["smem"]) +
              " ".join("%6d" % r[k] for k in COLS))


if __name__ == "__main__":
    main()
