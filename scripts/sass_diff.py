"""Per-kernel registers, spill bytes and SASS instruction counts of two builds of one .cu file, side by side.

Needs no GPU.  Compile each side to a cubin with the flags of pyflyt_drone_b200/build.py plus `-Xptxas -v -cubin`, keeping
ptxas' report, then:

    python scripts/sass_diff.py parent.cubin parent_ptxas.txt branch.cubin branch_ptxas.txt

Kernels are matched by their demangled name with the trailing `, false` template arguments a defaulted flag adds removed, so
that `fw_step_kernel<1, false, true>` (parent) and `fw_step_kernel<1, false, true, false>` (a build with an extra defaulted
template flag) compare as one row.  Kernels only one side has are listed apart.
"""
from __future__ import annotations

import re
import subprocess
import sys


def _demangle(names: list[str]) -> dict[str, str]:
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return dict(zip(names, out))


def _key(demangled: str) -> str:
    s = re.sub(r"\(.*\)$", "", demangled)                 # drop the parameter list
    s = re.sub(r"^void ", "", s).replace("<false>", "")
    while True:
        t = re.sub(r", false>", ">", s)
        if t == s:
            return s
        s = t


def sass_counts(cubin: str) -> dict[str, int]:
    txt = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    counts: dict[str, int] = {}
    cur = None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = 0
        elif cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+\S", line):
            counts[cur] += 1
    return counts


def ptxas_usage(log: str) -> dict[str, tuple[int, int, int]]:
    """mangled name -> (registers, spill stores, spill loads)"""
    res: dict[str, tuple[int, int, int]] = {}
    cur = None
    spills = (0, 0)
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            spills = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            res[cur] = (int(m.group(1)), *spills)
            spills = (0, 0)
    return res


def table(cubin: str, log: str) -> dict[str, tuple]:
    sc = sass_counts(cubin)
    us = ptxas_usage(log)
    dm = _demangle(list(sc))
    return {_key(dm[k]): (us.get(k, (-1, -1, -1)), v) for k, v in sc.items()}


def main() -> int:
    a = table(sys.argv[1], sys.argv[2])
    b = table(sys.argv[3], sys.argv[4])
    same = 0
    print("| kernel | regs | spill st/ld (B) | SASS instr. | parent -> branch |")
    print("|---|---|---|---|---|")
    for k in sorted(a):
        if k not in b:
            print(f"| `{k}` | missing on the branch | | | |")
            continue
        (ra, sa, la), ca = a[k]
        (rb, sb, lb), cb = b[k]
        eq = (ra, sa, la, ca) == (rb, sb, lb, cb)
        same += eq
        print(f"| `{k}` | {ra} -> {rb} | {sa}/{la} -> {sb}/{lb} | {ca} -> {cb} | {'identical' if eq else 'DIFFERS'} |")
    print(f"\n{same} of {len(a)} parent kernels identical in registers, spills and instruction count.\n")
    print("Only on the branch:\n")
    print("| kernel | regs | spill st/ld (B) | SASS instr. |")
    print("|---|---|---|---|")
    for k in sorted(set(b) - set(a)):
        (r, s, l), c = b[k]
        print(f"| `{k}` | {r} | {s}/{l} | {c} |")
    return 0


if __name__ == "__main__":
    sys.exit(main())
