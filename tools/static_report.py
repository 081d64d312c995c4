#!/usr/bin/env python
"""Static evidence that needs no GPU: per-kernel ptxas figures (registers, spills, static shared memory) from the
build's ptxas logs and SASS mnemonic counts from `cuobjdump -sass tol_b200/libtolcuda.so`.

    python tools/static_report.py [> profiles/rN_static_ptxas_sass.txt]

Template arguments of fg_cta_kernel<FORM, WIND, MAXT, PER, MODE, LOOP> / fg_long_kernel<FORM, WIND, MODE>:
FORM 7 = G7, 10 = S10; WIND 0 / 1 / 3; MODE 0 PLAIN, 1 SUMMARY, 2 COMPACT, 3 JVP, 4 VJP, 5 F only, 6 F only + summary
(fg_kernels.cu); fg_cta_goals_kernel / fg_long_goals_kernel are the same instances with a per-trajectory goal table;
fg_cta_hvp_kernel<FORM, WIND, MAXT, PER, LOOP> / fg_long_hvp_kernel<FORM, WIND> are MODE 7, the Hessian-of-the-Lagrangian
product (dual arithmetic)."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGS = [os.path.join(ROOT, "build", "csrc", f) for f in ("fg_kernels.ptxas.log", "expand_kernel.ptxas.log")]
LIB = os.path.join(ROOT, "tol_b200", "libtolcuda.so")
# mnemonics worth counting: the data path (TMA bulk copy, cp.async, fences), FP64 arithmetic, special functions
KEYS = ("UBLKCP", "LDGSTS", "FENCE", "MEMBAR", "SYNCS", "LDG", "STG", "LDS", "STS", "LDL", "STL", "DFMA", "DMUL", "DADD",
        "MUFU", "SHFL", "BAR", "WARPSYNC", "ATOMS", "LDC", "BRA")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    short = []
    for d in out[:len(names)]:
        d = re.sub(r"\(anonymous namespace\)::", "", d)
        d = re.sub(r"^void ", "", d)
        d = re.sub(r"\(FgConst.*$", "", d)
        d = re.sub(r"\((int|long|double|unsigned).*$", "", d)
        d = re.sub(r"\(int\)|\(bool\)", "", d)
        short.append(d)
    return short


def ptxas_table():
    rows = []
    for log in LOGS:
        if not os.path.exists(log):
            continue
        txt = open(log).read()
        for m in re.finditer(r"Compiling entry function '(\S+)' for '(\S+)'\n.*\n\s+(\d+) bytes stack frame, (\d+) bytes "
                             r"spill stores, (\d+) bytes spill loads\n.*Used (\d+) registers(?:, used (\d+) barriers)?"
                             r"(?:, (\d+) bytes cumulative stack size)?(?:, (\d+) bytes smem)?", txt):
            rows.append((m.group(1), m.group(2), int(m.group(6)), int(m.group(3)), int(m.group(4)), int(m.group(5)),
                         int(m.group(9) or 0)))
    return rows


def sass_counts():
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    per, cur = collections.OrderedDict(), None
    for ln in out.split("\n"):
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = per.setdefault(m.group(1), collections.Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", ln)
        if m and cur is not None:
            cur["_total"] += 1
            cur[m.group(1)] += 1
    return per


def main():
    rows = ptxas_table()
    names = demangle([r[0] for r in rows])
    print("# ptxas -v, sm_100a (build/csrc/*.ptxas.log): %d entry functions" % len(rows))
    print("%-62s %5s %6s %7s %7s %7s" % ("kernel", "regs", "stack", "spill_st", "spill_ld", "smem_static"))
    for r, nm in sorted(zip(rows, names), key=lambda t: t[1]):
        print("%-62s %5d %6d %7d %7d %7d" % (nm, r[2], r[3], r[4], r[5], r[6]))
    spilled = [nm for r, nm in zip(rows, names) if r[4] or r[5]]
    print("\nentry functions with spills: %d of %d" % (len(spilled), len(rows)))
    print("registers: min %d, max %d" % (min(r[2] for r in rows), max(r[2] for r in rows)))

    per = sass_counts()
    dn = dict(zip(per.keys(), demangle(list(per.keys()))))
    print("\n# cuobjdump -sass tol_b200/libtolcuda.so: instruction counts per kernel (static, not executed)")
    print("%-62s %6s " % ("kernel", "total") + " ".join("%6s" % k[:6] for k in KEYS))
    for k, cnt in sorted(per.items(), key=lambda t: dn[t[0]]):
        print("%-62s %6d " % (dn[k], cnt["_total"]) + " ".join("%6d" % cnt[m] for m in KEYS))
    wgmma = sum(1 for c in per.values() for m in c if m.startswith(("HGMMA", "WGMMA", "UTCHMMA", "HMMA")))
    print("\ntensor-core mnemonics anywhere in the library: %d (FP64 stencil-like map; none expected)" % wgmma)
    with_tma = sum(1 for c in per.values() if c["UBLKCP"])
    print("kernels that issue TMA bulk copies (UBLKCP): %d of %d; with cp.async (LDGSTS): %d" % (
        with_tma, len(per), sum(1 for c in per.values() if c["LDGSTS"])))


if __name__ == "__main__":
    sys.exit(main())
