#!/usr/bin/env python
"""Kernel-by-kernel SASS comparison of two builds of the same object:
    tools/sass_compare.py <a.o> <b.o>
cuobjdump prints each __global__ function (with its inlined copies of the __noinline__ helpers) as a
section of its own; addresses and encodings are dropped, the rest is compared section by section.
Under the arithmetic contract (ttmpc_device.cuh) a refactor that leaves a kernel byte-identical here
cannot have changed its results.  Exit status 1 when any kernel differs or exists in one build only."""
import re
import subprocess
import sys


def kernels(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = d.setdefault(m.group(1), [])
        elif cur is not None:
            s = re.sub(r"/\*[0-9a-f]{4,}\*/|/\* 0x[0-9a-f]+ \*/", "", line).strip()
            if s:
                cur.append(s)
    return d


a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
differ = [k for k in a if k in b and a[k] != b[k]]
print("kernels: %d and %d, identical %d, differ %d" % (len(a), len(b), sum(a[k] == b.get(k) for k in a), len(differ)))
for tag, names in (("only in a", sorted(set(a) - set(b))), ("only in b", sorted(set(b) - set(a))), ("differ", differ)):
    for k in names:
        print("  %s: %s" % (tag, k) + ("  (%d / %d instructions)" % (len(a[k]), len(b[k])) if tag == "differ" else ""))
sys.exit(1 if differ or set(a) != set(b) else 0)
