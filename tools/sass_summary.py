"""SASS evidence of the shipped library: per kernel - registers, stack, shared memory, instruction count, TMA / mbarrier
sites (UBLKCP / SYNCS), local-memory traffic (STL / LDL), global store widths, FP64 and MUFU counts.

    python tools/sass_summary.py [lib.so] > profiles/r02_sass_summary.md
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "ray-tracer-engine_b200", "libore_b200.so")


def demangle(name):
    try:
        return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip() or name
    except Exception:
        return name


res = {}
cur = None
for line in subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout.splitlines():
    m = re.search(r"Function (\S+):", line)
    if m:
        cur = m.group(1)
        continue
    m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", line)
    if m and cur:
        res[cur] = tuple(int(v) for v in m.groups())
        cur = None

sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
arch = sorted(set(re.findall(r"arch = (sm_\w+)", sass)))
kern = collections.OrderedDict()
cur = None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1)
        kern[cur] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
    if m and cur:
        op = m.group(1)
        c = kern[cur]
        c["total"] += 1
        base = op.split(".")[0]
        c[base] += 1
        if base == "STG":
            c["STG." + ("128" if ".128" in op else "64" if ".64" in op else "32")] += 1
        if base == "LDG":
            c["LDG." + ("128" if ".128" in op else "64" if ".64" in op else "32")] += 1
        if base in ("LDS", "STS"):
            c[base + "." + ("128" if ".128" in op else "64" if ".64" in op else "32")] += 1

print("# SASS summary of the shipped library (round 2)\n")
print(f"`{os.path.relpath(lib, ROOT)}`: {os.path.getsize(lib) / 1e6:.1f} MB, cubin architectures: {', '.join(arch)} "
      f"(cuobjdump -sass / -res-usage; produced by `tools/sass_summary.py`).\n")
print("TMA bulk copies (`cp.async.bulk`) appear as `UBLKCP`, mbarrier operations as `SYNCS`; `STL`/`LDL` are local-memory "
      "(stack) accesses; `D*` are FP64 instructions (the double-precision islands of the reference's arithmetic); "
      "there are no tensor-core (`UTC*MMA`, `HMMA`) or TMEM (`LDTM`/`STTM`) instructions: the path is scalar FP32 tests, "
      "not a contraction.\n")
print("| kernel | regs | stack B | SASS instr | UBLKCP | SYNCS | STL | LDL | STG 32/64/128 | LDG 32/64/128 | LDS | FP64 (DADD+DMUL+DFMA+DSETP) | MUFU | UTC*MMA/HMMA |")
print("|---|---|---|---|---|---|---|---|---|---|---|---|---|---|")
for k, c in kern.items():
    # FAST_LIBM instantiations (last template argument true): only those of the default path are listed
    if k.startswith("_ZN3ore") and "Lb1EEEv" in k and not any(
            s in k for s in ("primary_tile_kernelILi8ELb0ELb1", "shadow_sweep_kernelILb0ELb1ELb1", "shade_setup")):
        continue
    r = res.get(k, (0, 0, 0, 0))
    name = demangle(k).replace("ore::", "").replace("void ", "")
    fp64 = c["DADD"] + c["DMUL"] + c["DFMA"] + c["DSETP"]
    tc = sum(v for kk, v in c.items() if kk.startswith("UTC") or kk in ("HMMA", "LDTM", "STTM"))
    print(f"| `{name}` | {r[0]} | {r[1]} | {c['total']} | {c['UBLKCP']} | {c['SYNCS']} | {c['STL']} | {c['LDL']} | "
          f"{c['STG.32']}/{c['STG.64']}/{c['STG.128']} | {c['LDG.32']}/{c['LDG.64']}/{c['LDG.128']} | {c['LDS']} | {fp64} | {c['MUFU']} | {tc} |")
print("\n(The last template argument of the three render kernels is `FAST_LIBM`: `true` = CUDA's libm for "
      "`ORE_FLAG_FAST_LIBM`; only the default-path instantiations of it are listed.)")
