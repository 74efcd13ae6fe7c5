#!/usr/bin/env python
"""profiles/sass_same.py <objdir A> <objdir B> — which kernels' SASS differs between two builds of rala_b200/csrc
(e.g. rala_b200/build/<variant>/ against rala_b200/build/, or the parent commit's build against this one).  Used when
code is added behind a switch, or a settled switch is removed: the kernels of the default path must come out
bit-identical to the build that was tested."""
import hashlib
import re
import subprocess
import sys


def funcs(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            res[cur].append(re.sub(r"/\* 0x[0-9a-f]+ \*/", "", line).strip())
    return {k: hashlib.md5("\n".join(v).encode()).hexdigest() for k, v in res.items()}


a_dir, b_dir = sys.argv[1], sys.argv[2]
rc = 0
for f in ("classify", "containment", "graph_build", "transitive", "fabric", "frontend"):   # every object with kernels
    a, b = funcs(f"{a_dir}/{f}.o"), funcs(f"{b_dir}/{f}.o")
    changed = sorted(k for k in a if k in b and a[k] != b[k])
    print(f"{f}: {len(a)} / {len(b)} kernels, changed: {changed or 'none'}, only in A: {sorted(set(a) - set(b)) or 'none'}, "
          f"only in B: {sorted(set(b) - set(a)) or 'none'}")
    rc |= bool(changed)
sys.exit(rc)
