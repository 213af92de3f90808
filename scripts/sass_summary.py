#!/usr/bin/env python
"""Per-kernel SASS evidence of the Blackwell/Hopper-native data movement in libspmv_b200.so:
UBLKCP = cp.async.bulk (1-D TMA bulk copy), SYNCS = mbarrier operations, SHFL = warp shuffles;
registers from cuobjdump -res-usage.      python scripts/sass_summary.py > profiles/sass_summary.txt

shipped_kernels() and short_name() are also the kernel list of tests/test_gpu_kernel_coverage.py."""
import os
import re
import subprocess
import sys

LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "gpu-spmv_b200", "lib", "libspmv_b200.so")


def short_name(demangled):
    """`void (anonymous namespace)::k<1, 2>(int, float*)` -> `k<1, 2>`: no return type, no namespace of the
    library, no parameter list; `> >` is written `>>` (c++filt and CUPTI spell nested templates differently)."""
    d = demangled.replace("(anonymous namespace)::", "").replace("spmv::b200::", "").strip()
    d = re.sub(r"^void ", "", d)
    depth, cut = 0, len(d)
    for i, ch in enumerate(d):  # cut at the parameter list: the first '(' outside template brackets
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            cut = i
            break
    return re.sub(r">\s+>", ">>", d[:cut])


def demangle(names):
    """Short names of kernel symbols, mangled or already demangled, in order."""
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return [short_name(d) for d in out.splitlines()]


def kernel_registers(lib=LIB):
    """Mangled name -> registers of every kernel in the library's cubins (cuobjdump -res-usage)."""
    res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    regs, cur = {}, None
    for line in res.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            cur = m.group(1)
            regs.setdefault(cur, "?")
        m = re.search(r"REG:(\d+)", line)
        if m and cur:
            regs[cur] = int(m.group(1))
    return regs


def shipped_kernels(lib=LIB):
    """The short names of every kernel the library ships."""
    return set(demangle(list(kernel_registers(lib))))


def main(lib=LIB):
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    regs = kernel_registers(lib)
    rows, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            rows[cur] = dict(n=0, UBLKCP=0, SYNCS=0, LDG=0, LDS=0, STG=0, SHFL=0, ATOM=0)
            continue
        if cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
            r = rows[cur]
            r["n"] += 1
            for k in ("UBLKCP", "SYNCS", "LDG", "LDS", "STG", "SHFL"):
                if re.search(r"\b" + k, line):
                    r[k] += 1
            if re.search(r"\b(ATOM|RED)\b|\bATOMG|\bREDG|\bATOMS", line):
                r["ATOM"] += 1
    names = list(rows)
    short = demangle(names)
    arch = sorted(set(re.findall(r"sm_\d+a?", subprocess.run(["cuobjdump", "-lelf", lib], capture_output=True, text=True).stdout)))
    print(f"# libspmv_b200.so: {len(names)} kernels, cubin architectures {arch}")
    print("# kernel | SASS instructions | registers | UBLKCP (TMA bulk copy) | SYNCS (mbarrier) | LDG | LDS | STG | SHFL | ATOM/RED")
    tot = dict(UBLKCP=0, SYNCS=0)
    for name, s in sorted(zip(names, short), key=lambda t: t[1]):
        r = rows[name]
        tot["UBLKCP"] += r["UBLKCP"]
        tot["SYNCS"] += r["SYNCS"]
        print(f"{s} | {r['n']} | {regs.get(name, '?')} | {r['UBLKCP']} | {r['SYNCS']} | {r['LDG']} | {r['LDS']} | {r['STG']} | {r['SHFL']} | {r['ATOM']}")
    print(f"# total UBLKCP {tot['UBLKCP']}, SYNCS {tot['SYNCS']}")
    ptx_like = len(re.findall(r"multimem|MULTIMEM", sass))
    print(f"# multimem (NVSwitch multicast) instructions visible in SASS: {ptx_like} (a multimem.st is a plain store to a multicast-mapped address at SASS level)")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else LIB)
