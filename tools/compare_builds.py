#!/usr/bin/env python3
"""tools/compare_builds.py OLD_LIB NEW_LIB OLD_PTXAS_LOG NEW_PTXAS_LOG [OUT] [OLD_KERNEL=NEW_KERNEL ...] -- registers, spills
and SASS of every kernel of two builds of a library side by side (no GPU needed).

The logs are the `-Xptxas -v` output of `python -m audiosdr_b200.build --force` for each build; the SASS comes from
`cuobjdump -sass` of the libraries.  Kernels are matched by mangled name; an OLD_KERNEL=NEW_KERNEL pair matches a kernel that
was renamed (for example a twin that became a template instantiation).  A matched kernel is the same when its registers and
spills are, and when its instructions are, each compared as text and encoding (control bits included) with the address
removed.  Prints (and writes to OUT) one line per kernel, the list of kernels that differ and the list of kernels only the
new build has."""
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


def sass(lib):
    """kernel -> list of its instructions, each `text ; /* encoding */ /* encoding */` with the address stripped"""
    txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    n, fn = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
            n[fn] = []
            continue
        if not fn:
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(\S.*)", line)
        if m:
            n[fn].append(" ".join(m.group(1).split()))
        elif n[fn] and re.match(r"\s+/\* 0x[0-9a-f]+ \*/\s*$", line):  # second encoding word of the instruction above
            n[fn][-1] += " " + line.strip()
    return n


def main():
    args = sys.argv[1:]
    old_lib, new_lib, old_log, new_log = args[:4]
    rest = args[4:]
    pairs = dict(a.split("=", 1) for a in rest if "=" in a)
    out = [a for a in rest if "=" not in a]
    po, pn, so, sn = ptxas(old_log), ptxas(new_log), sass(old_lib), sass(new_lib)
    renamed = set(pairs.values())
    rows = [(o, pairs.get(o, o)) for o in so] + [(None, n) for n in sn if n not in renamed and n not in so]
    lines, differ, added = [], [], []
    lines.append("%-44s %14s %14s %18s %10s" % ("kernel", "regs old/new", "spill old/new", "SASS instr old/new", "SASS code"))
    for o, n in sorted(rows, key=lambda r: r[1]):
        a, b = po.get(o, {}), pn.get(n, {})
        io, inew = so.get(o), sn.get(n)
        text = "-" if io is None or inew is None else ("same" if io == inew else "differs")
        row = (n, "%s/%s" % (a.get("regs"), b.get("regs")), "%s|%s" % (a.get("spill"), b.get("spill")),
               "%s/%s" % (io and len(io), inew and len(inew)), text)
        same = a == b and text == "same"
        line = "%-44s %14s %14s %18s %10s" % row
        if o is not None and o != n:
            line += "   (old: %s)" % o
        if o is None:
            lines.append(line + "   NEW")
            added.append(n)
            continue
        lines.append(line + ("" if same else "   DIFFERS"))
        if not same:
            differ.append(n if inew is not None else o)
    lines.append("")
    lines.append("kernels that differ: %s" % (", ".join(differ) if differ else "none"))
    lines.append("kernels only in the new build: %s" % (", ".join(added) if added else "none"))
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if out:
        with open(out[0], "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
