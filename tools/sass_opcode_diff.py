"""Opcode histogram of every kernel in two builds of one translation unit, side by side. Usage:
  nvcc <the flags of build.py> -cubin -o before.cubin csrc/k_narrow.cu     (at the old commit)
  nvcc <the flags of build.py> -cubin -o after.cubin csrc/k_narrow.cu      (at the new one)
  python tools/sass_opcode_diff.py before.cubin after.cubin [kernel name substring]
Prints, per kernel present in both, "same" or the opcodes whose counts differ. Operands (register
numbers, constant-bank offsets, branch targets) are not compared: a change that only moves data
leaves the histogram alone, one that adds or removes work does not."""
import collections
import re
import subprocess
import sys


def histograms(cubin):
    out = subprocess.run(["cuobjdump", "-sass", cubin], check=True, capture_output=True, text=True).stdout
    hist, cur = {}, None
    for ln in out.split("\n"):
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            hist[cur] = collections.Counter()
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", ln)
        if m and cur is not None:
            hist[cur][m.group(2)] += 1
    return hist


def main():
    a, b = histograms(sys.argv[1]), histograms(sys.argv[2])
    sub = sys.argv[3] if len(sys.argv) > 3 else ""
    for k in sorted(set(a) | set(b)):
        if sub not in k:
            continue
        if k not in a or k not in b:
            print("%-8s %s" % ("only-" + ("new" if k in b else "old"), k))
            continue
        diff = {op: (a[k][op], b[k][op]) for op in set(a[k]) | set(b[k]) if a[k][op] != b[k][op]}
        total = sum(b[k].values())
        print("%-8s %6d instr  %s" % ("same" if not diff else "DIFFERS", total, k))
        for op, (x, y) in sorted(diff.items()):
            print("           %-16s %6d -> %6d" % (op, x, y))


if __name__ == "__main__":
    main()
