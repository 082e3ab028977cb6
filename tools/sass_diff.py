#!/usr/bin/env python
"""Compares the SASS of two builds function by function (cuobjdump -sass; runs without a GPU).

    python tools/sass_diff.py LIB_A LIB_B

Prints every function as `same` or `DIFF` with the number of differing instruction lines (addresses and encodings
included), and `only in A` / `only in B` for a function one side lacks.  Exits 1 if any function differs or is missing on one
side.  cuobjdump -sass prints no line info, so code that only moved in the source compares equal.
"""
import collections
import difflib
import re
import subprocess
import sys


def functions(lib):
    """{name: [instruction lines]}; a name that occurs in several cubins gets a #k suffix from its second occurrence on."""
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, seen, cur = {}, collections.Counter(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            seen[name] += 1
            cur = name if seen[name] == 1 else f"{name}#{seen[name]}"
            out[cur] = []
        elif cur is not None and line.strip().startswith("/*"):
            out[cur].append(line.strip())
    return out


def differing_lines(a, b):
    sm = difflib.SequenceMatcher(None, a, b, autojunk=False)
    return sum(max(i2 - i1, j2 - j1) for op, i1, i2, j1, j2 in sm.get_opcodes() if op != "equal")


def main(argv):
    if len(argv) != 3:
        print(__doc__.strip(), file=sys.stderr)
        return 2
    fa, fb = functions(argv[1]), functions(argv[2])
    bad = 0
    for name in sorted(fa.keys() | fb.keys()):
        if name not in fb:
            print(f"only in A  {name}")
        elif name not in fa:
            print(f"only in B  {name}")
        elif fa[name] == fb[name]:
            print(f"same       {name}")
            continue
        else:
            print(f"DIFF {differing_lines(fa[name], fb[name]):5d}  {name}")
        bad += 1
    print(f"{len(fa.keys() | fb.keys()) - bad} same, {bad} differing or missing")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
