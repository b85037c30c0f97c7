#!/usr/bin/env python3
"""Check that a change leaves the machine code of existing kernels alone.

    python tools/sass_compare.py OLD.so NEW.so

Disassembles both libraries with `cuobjdump -sass`, splits the listing into functions and compares every function of
OLD with the function of the same mangled name in NEW, instruction for instruction.  Anonymous-namespace names are
compared without the per-build hash nvcc puts in them.  A name that several translation units define (a static kernel
of a shared header) is compared as the multiset of its bodies.  Prints one line per function of OLD that is missing
from NEW or differs, then the functions only NEW has, and exits 1 if any OLD function is missing or differs.  A kernel
that gained a template parameter has a new name: compare its old and new instantiations by hand
(`cuobjdump -sass -fun NAME`).
"""
import collections
import re
import subprocess
import sys


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    # nvcc names a translation unit's anonymous namespace with a hash of where it was built
    out = re.sub(r"_GLOBAL__N__[0-9a-f]{8}_", "_GLOBAL__N__", out)
    funcs, name, body = collections.defaultdict(list), None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m or re.match(r"\s*(Fatbin|code for sm_)", line):
            if name:
                funcs[name].append("\n".join(body))
            name, body = (m.group(1) if m else None), []
            continue
        if name and line.strip():
            body.append(line.strip())
    if name:
        funcs[name].append("\n".join(body))
    return {k: sorted(v) for k, v in funcs.items()}


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    bad = 0
    for name in sorted(old):
        if name not in new:
            print("missing  ", name)
            bad += 1
        elif old[name] != new[name]:
            print("differs  ", name)
            bad += 1
    added = sorted(set(new) - set(old))
    print("%d functions in the old library, %d missing or different; %d only in the new one%s"
          % (len(old), bad, len(added), (": " + " ".join(added)) if added else ""))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
