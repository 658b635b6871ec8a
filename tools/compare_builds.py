#!/usr/bin/env python3
"""tools/compare_builds.py OLD_LIB NEW_LIB OLD_PTXAS_LOG NEW_PTXAS_LOG [OUT] -- registers, spills and SASS instruction counts of
every kernel of two builds of libsdr_batch.so side by side (no GPU needed).

The logs are the `-Xptxas -v` output of `python -m audiosdr_b200.build --force` for each build; the instruction counts come from
`cuobjdump -sass` of the libraries.  Prints (and writes to OUT) one line per kernel and the list of kernels that differ."""
import collections
import re
import subprocess
import sys


def ptxas(log):
    out, fn = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            fn = m.group(1)
            out[fn] = {}
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and fn:
            out[fn]["spill"] = "%s/%s" % m.groups()
        m = re.search(r"Used (\d+) registers", line)
        if m and fn:
            out[fn]["regs"] = int(m.group(1))
    return out


def sass_counts(lib):
    txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    n, fn = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
            n[fn] = 0
            continue
        if fn and re.match(r"\s+/\*[0-9a-f]+\*/\s+\S", line):
            n[fn] += 1
    return n


def main():
    old_lib, new_lib, old_log, new_log = sys.argv[1:5]
    po, pn, so, sn = ptxas(old_log), ptxas(new_log), sass_counts(old_lib), sass_counts(new_lib)
    lines, differ = [], []
    lines.append("%-44s %14s %14s %18s" % ("kernel", "regs old/new", "spill old/new", "SASS instr old/new"))
    for fn in sorted(set(so) | set(sn)):
        a, b = po.get(fn, {}), pn.get(fn, {})
        row = (fn, "%s/%s" % (a.get("regs"), b.get("regs")), "%s|%s" % (a.get("spill"), b.get("spill")), "%s/%s" % (so.get(fn), sn.get(fn)))
        same = a == b and so.get(fn) == sn.get(fn)
        lines.append("%-44s %14s %14s %18s%s" % (row + ("" if same else "   DIFFERS",)))
        if not same:
            differ.append(fn)
    lines.append("")
    lines.append("kernels that differ: %s" % (", ".join(differ) if differ else "none"))
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if len(sys.argv) > 5:
        with open(sys.argv[5], "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
