#!/usr/bin/env python
"""Compare the SASS of every kernel two builds of the library have in common (matched by mangled symbol name; addresses
and encodings stripped).  Usage: python tools/sass_compare.py OLD.so NEW.so"""
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    res, name, lines = {}, None, []
    for ln in out.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            if name:
                res[name] = lines
            name, lines = m.group(1), []
        elif re.match(r"\s*/\*[0-9a-f]{4,}\*/", ln):  # instruction lines (offsets grow past 4 hex digits)
            lines.append(re.sub(r"/\* 0x[0-9a-f]+ \*/", "", re.sub(r"^\s*/\*[0-9a-f]{4,}\*/", "", ln)).strip())
    if name:
        res[name] = lines
    return res


old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
for k in sorted(set(old) | set(new)):
    if k not in old:
        verdict = "new"
    elif k not in new:
        verdict = "removed"
    else:
        verdict = "IDENTICAL" if old[k] == new[k] else "differs (%d -> %d instructions)" % (len(old[k]), len(new[k]))
    print("%-90s %6d instructions  %s" % (k, len(new.get(k, old.get(k))), verdict))
