#!/usr/bin/env python3
"""Per-kernel SASS comparison of two builds of the library: every kernel of every object file (cuobjdump -sass), with addresses
and the encoding words dropped, compared by mangled name (anonymous-namespace tags removed). Prints one line per kernel (same / changed / added / removed) and a total.

    python scratch/sass_diff.py <build dir A> <build dir B>     # e.g. a build of the parent commit and software-raytracer_b200/build
"""
import os
import re
import subprocess
import sys


def kernels(obj):
    """{mangled name: [instruction text, ...]} of one object file."""
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__\w+?_cu_[0-9a-f]{8}", "_GLOBAL__N_", m.group(1))   # the anonymous namespace's per-build tag
            res[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if cur and m:
            res[cur].append(m.group(1))
    return res


def main(a_dir, b_dir):
    objs = sorted(f for f in os.listdir(b_dir) if f.endswith(".o"))
    counts = {"same": 0, "changed": 0, "added": 0, "removed": 0}
    for o in objs:
        a = kernels(os.path.join(a_dir, o)) if os.path.exists(os.path.join(a_dir, o)) else {}
        b = kernels(os.path.join(b_dir, o))
        for name in sorted(set(a) | set(b)):
            if name not in a:
                st = "added"
            elif name not in b:
                st = "removed"
            else:
                st = "same" if a[name] == b[name] else "changed"
            counts[st] += 1
            n = len(b.get(name, a.get(name)))
            print("%-8s %-16s %6d  %s" % (st, o, n, name))
    print("kernels: %d same, %d changed, %d added, %d removed" % (counts["same"], counts["changed"], counts["added"], counts["removed"]))
    return 1 if counts["changed"] or counts["removed"] else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
