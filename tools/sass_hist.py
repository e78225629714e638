#!/usr/bin/env python
"""SASS instruction histogram of kernels in a cubin-carrying binary (no GPU needed):

    python tools/sass_hist.py zk_stark_project_b200/libzkb200.so k_ntt_pass k_hash_lde_rows ... > profiles/rN_sass_hist.txt

For every kernel whose mangled name contains one of the patterns it prints the opcode histogram, the split into FMA-pipe
(IMAD*) / ALU-pipe / memory classes and — when the kernel has one dominant backward branch — the same for its hottest loop.

    python tools/sass_hist.py --regions BINARY KERNEL label=LO-HI[*N][+LO-HI[*N]..] ...

counts the instructions a thread executes per kernel invocation, region by region: each region is a list of SASS address ranges
[LO, HI) (hex, as printed by cuobjdump -sass) on the path the thread takes, each weighted by how often it runs (loop trips).
The ranges are read off the disassembly of one build for one launch shape and have to be re-read after any change of the kernel."""
import collections
import re
import subprocess
import sys


def kernels(binary):
    out = subprocess.check_output(["cuobjdump", "-sass", binary], text=True)
    cur, body = None, []
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            if cur:
                yield cur, body
            cur, body = m.group(1), []
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and cur:
            body.append((int(m.group(1), 16), m.group(2).strip()))
    if cur:
        yield cur, body


def opcode(ins):
    ins = re.sub(r"^@!?U?P\w+\s+", "", ins)
    return ins.split()[0] if ins else "?"


def classes(ops):
    c = collections.Counter()
    for o in ops:
        if o.startswith("IMAD.WIDE"):
            c["IMAD.WIDE (FMA pipe)"] += 1
        elif o.startswith("IMAD.HI"):
            c["IMAD.HI (FMA pipe, half rate)"] += 1
        elif o.startswith("IMAD"):
            c["other IMAD: MOV/IADD/X/lo (FMA pipe)"] += 1
        elif re.match(r"(IADD3|VIADD|SEL|LOP3|PLOP3|SHF|PRMT|ISETP|LEA|IABS|FLO|POPC|BREV|VOTE|UIADD3|ULOP3|USHF|UPRMT|USEL|UISETP)", o):
            c["ALU / uniform pipe"] += 1
        elif re.match(r"(LDG|STG|LDS|STS|LDC|LDCU|ATOM|RED|LDL|STL|SHFL|UTMA|UBLK)", o):
            c["memory / shuffle"] += 1
        else:
            c["control / other"] += 1
    return c


def report(name, body):
    ops = [opcode(i) for _, i in body if not i.startswith("NOP")]
    print(f"== {name}: {len(ops)} instructions")
    for k, v in classes(ops).most_common():
        print(f"   {v:6d}  {k}")
    print("   top opcodes: " + ", ".join(f"{o} {n}" for o, n in collections.Counter(ops).most_common(14)))
    best = None
    addr = [a for a, _ in body]
    for idx, (a, i) in enumerate(body):
        m = re.search(r"BRA(?:\.U)?\s+.*?(0x[0-9a-f]+)\s*$", i)
        if m:
            t = int(m.group(1), 16)
            if t < a and t in addr:
                s = addr.index(t)
                if best is None or idx - s > best[1] - best[0]:
                    best = (s, idx)
    if best and best[1] - best[0] > 64:
        lops = [opcode(i) for _, i in body[best[0]:best[1] + 1]]
        print(f"   largest loop: {len(lops)} instructions: " + "; ".join(f"{v} {k}" for k, v in classes(lops).most_common()))


def regions(binary, kernel, specs):
    body = next((b for n, b in kernels(binary) if n == kernel), None)
    if body is None:
        sys.exit(f"no kernel {kernel} in {binary}")
    total = 0
    print(f"== {kernel}: instructions per thread and invocation, by region")
    for spec in specs:
        label, ranges = spec.split("=", 1)
        n = 0
        for r in ranges.split("+"):
            span, _, mult = r.partition("*")
            lo, hi = (int(x, 16) for x in span.split("-"))
            n += sum(1 for a, i in body if lo <= a < hi and not i.startswith("NOP")) * (int(mult) if mult else 1)
        total += n
        print(f"   {n:6d}  {label}  ({ranges})")
    print(f"   {total:6d}  total")


if __name__ == "__main__":
    if sys.argv[1] == "--regions":
        regions(sys.argv[2], sys.argv[3], sys.argv[4:])
        sys.exit(0)
    binary, pats = sys.argv[1], sys.argv[2:]
    for name, body in kernels(binary):
        if any(p in name for p in pats):
            report(name, body)
