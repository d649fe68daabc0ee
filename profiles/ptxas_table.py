"""Registers, stack and spill bytes per kernel from `nvcc -Xptxas -v` output (python -m
physicsbasedbayesianinference_b200.build --force -v 2> log), and the comparison of two such logs.

    python profiles/ptxas_table.py LOG [--grep SUBSTRING]             one line per kernel instance
    python profiles/ptxas_table.py BEFORE AFTER [--grep SUBSTRING]    instances whose numbers differ, and the count of
                                                                      instances present in both / only in AFTER

Instances are matched by demangled name.  k_small_run gained a template flag TEMPER and a TemperRun argument (the
tempered run); an untempered instance k_small_run<..., false>(..., ehmc::TemperRun) of AFTER is matched with
k_small_run<...>(...) of BEFORE.
"""
from __future__ import annotations

import re
import subprocess
import sys


def parse(path):
    """{mangled kernel name: (registers, stack frame bytes, spill store bytes, spill load bytes)}"""
    out, name, frame = {}, None, None
    for line in open(path):
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            name, frame = m.group(1), None
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            frame = tuple(int(x) for x in m.groups())
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out[name] = (int(m.group(1)),) + (frame or (0, 0, 0))
            name = None
    return out


def demangle(names):
    try:
        res = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
        return res.stdout.splitlines()
    except (OSError, subprocess.CalledProcessError):
        return list(names)


def canonical(name):
    """The demangled name with k_small_run's TEMPER = false flag and TemperRun argument removed."""
    name = re.sub(r"^(void ehmc::k_small_run<.*), false>\(", r"\1>(", name)
    return name.replace(", ehmc::TemperRun)", ")")


def main(argv):
    grep = None
    if "--grep" in argv:
        i = argv.index("--grep")
        grep = argv[i + 1]
        argv = argv[:i] + argv[i + 2:]
    logs = [parse(p) for p in argv]
    if len(logs) == 1:
        names = sorted(n for n in logs[0] if grep is None or grep in n)
        for n, d in zip(names, demangle(names)):
            r, f, s, l = logs[0][n]
            print(f"{r:4d} regs {f:6d} B stack {s:6d} B spill st {l:6d} B spill ld  {d}")
        return 0
    before, after = ({canonical(d): v for d, v in zip(demangle(list(log)), log.values())} for log in logs)
    common = sorted(n for n in before if n in after and (grep is None or grep in n))
    new = sorted(n for n in after if n not in before and (grep is None or grep in n))
    changed = [n for n in common if before[n] != after[n]]
    print(f"{len(common)} instances in both logs, {len(changed)} differ; {len(new)} only in the second log")
    for n in changed:
        print(f"  {before[n]} -> {after[n]}  {n}")
    return 1 if changed else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
