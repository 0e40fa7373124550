#!/usr/bin/env python3
"""Function-by-function comparison of the SASS of two builds of liblogmel_b200.so (no GPU needed):

    python tools/sass_compare.py OLD.so NEW.so

For every kernel of either file: whether its instructions are byte-identical, the instruction counts, the number of
differing lines when they are not, and the register / stack / spill figures ptxas reports (cuobjdump -res-usage).
Instruction lines are compared with their addresses and encodings stripped, so a function that only moved in the
file still counts as identical.  A kernel whose parameter list changed is paired with its namesake when each file has one
function of that name."""
from __future__ import annotations

import re
import shutil
import subprocess
import sys
from difflib import SequenceMatcher


def _cuobjdump() -> str:
    return shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def sass_functions(so: str) -> dict:
    text = subprocess.run([_cuobjdump(), "-sass", so], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if name and m:
            funcs[name].append(re.sub(r"\s+", " ", m.group(1)).strip())
    return funcs


def resources(so: str) -> dict:
    text = subprocess.run([_cuobjdump(), "-res-usage", so], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", line)
        if name and m:
            res[name] = (int(m.group(1)), int(m.group(2)))
    return res


def demangle(names) -> dict:
    cxx = shutil.which("c++filt") or shutil.which("cu++filt")
    if not cxx:
        return {n: n for n in names}
    out = subprocess.run([cxx], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def main(old: str, new: str) -> int:
    a, b = sass_functions(old), sass_functions(new)
    ra, rb = resources(old), resources(new)
    names = sorted(set(a) | set(b))
    pretty = demangle(names)
    base = lambda n: pretty[n].split("(")[0]
    renamed = {}   # new name -> old name of the same kernel with another parameter list
    for n in set(b) - set(a):
        old_n = [m for m in set(a) - set(b) if base(m) == base(n)]
        if len(old_n) == 1 and sum(base(m) == base(n) for m in b) == 1:
            renamed[n] = old_n[0]
    same = 0
    for n in names:
        if n in renamed.values():
            continue
        fa, fb = a.get(renamed.get(n, n)), b.get(n)
        if n in renamed:
            ra[n] = ra[renamed[n]]
            print(f"parameters changed: {pretty[renamed[n]]} -> {pretty[n]}")
        reg = f"regs {ra.get(n, ('-', '-'))[0]} -> {rb.get(n, ('-', '-'))[0]}, stack {ra.get(n, ('-', '-'))[1]} -> {rb.get(n, ('-', '-'))[1]}"
        if fa is None or fb is None:
            print(f"{'only in new' if fa is None else 'only in old'}: {pretty[n]}  ({reg})")
            continue
        if fa == fb:
            same += 1
            print(f"identical ({len(fa)} instructions, {reg}): {pretty[n]}")
            continue
        diff = sum(max(i2 - i1, j2 - j1) for tag, i1, i2, j1, j2 in SequenceMatcher(None, fa, fb, autojunk=False).get_opcodes()
                   if tag != "equal")
        print(f"DIFFERS ({len(fa)} -> {len(fb)} instructions, {diff} lines differ, {reg}): {pretty[n]}")
    print(f"{same} of {len(names) - len(renamed)} functions identical")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
