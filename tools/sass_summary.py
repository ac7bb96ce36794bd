"""Per-kernel SASS mnemonic counts of the built library -> profiles/<tag>_sass_summary.txt (the evidence
that the tcgen05 / TMEM / TMA / shared-atomic claims of DESIGN.md are in the shipped code).
    python tools/sass_summary.py [tag]        # default r2"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "articulation3d_b200", "csrc", "liba3d.so")
tag = sys.argv[1] if len(sys.argv) > 1 else "r2"
WATCH = ["UTCOMMA", "UTCIMMA", "UTCHMMA", "UTCQMMA", "LDTM", "STTM", "UTCBAR", "UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "POPC", "ATOMS", "RED",
         "ATOMG", "MUFU.RCP", "FFMA", "FFMA2", "DFMA", "DMUL", "DADD", "LOP3", "IMAD", "SHF", "FSETP", "LDS", "STS",
         "LDG", "STG", "REDUX", "BAR", "ACQBULK", "PREEXIT"]

sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
res = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
kernels, cur = collections.OrderedDict(), None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1)
        kernels[cur] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", line)
    if m and cur:
        op = m.group(1)
        kernels[cur]["_total"] += 1
        for w in WATCH:
            if op == w or op.startswith(w + "."):
                kernels[cur][w] += 1


def demangle(n):
    out = subprocess.run(["cu++filt", n], capture_output=True, text=True).stdout.strip()
    out = re.sub(r"\(anonymous namespace\)::|<unnamed>::", "", out)
    depth = 0
    for i, ch in enumerate(out):                 # cut the argument list: first '(' outside template brackets
        depth += ch == "<"
        depth -= ch == ">"
        if ch == "(" and depth == 0:
            return out[:i]
    return out


usage = {}
for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) .*?SHARED:(\d+)", res):
    usage[m.group(1)] = (int(m.group(2)), int(m.group(3)))
lines = [f"# SASS mnemonic counts per kernel of articulation3d_b200/csrc/liba3d.so (cuobjdump -sass, sm_100a), {tag}",
         "# UTCOMMA = tcgen05.mma kind::mxf4, LDTM = tcgen05.ld, UTCBAR = tcgen05.commit, UTMALDG = TMA tensor load, "
         "ATOMS/RED = shared / global atomics", ""]
for k, c in kernels.items():
    reg, sh = usage.get(k, (None, None))
    lines.append(f"{demangle(k)}   [{c['_total']} instructions, {reg} regs, {sh} B static smem]")
    lines.append("    " + "  ".join(f"{w}={c[w]}" for w in WATCH if c[w]))
out = os.path.join(ROOT, "profiles", f"{tag}_sass_summary.txt")
with open(out, "w") as f:
    f.write("\n".join(lines) + "\n")
print(out)
print("\n".join(lines[:12]))
