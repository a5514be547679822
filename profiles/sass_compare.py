"""Kernel-by-kernel comparison of two builds' SASS (cuobjdump -sass of every object in build/):
    python profiles/sass_compare.py <parent build dir> <this build dir> [old=new ...]
Addresses and the comment columns are dropped, so a kernel reads "identical" when its instruction stream is.  Each
old=new replaces a substring of the parent's kernel names, to pair a kernel with its renamed successor (a new template
parameter, an appended kernel parameter)."""
import collections
import os
import re
import subprocess
import sys


def kernels(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    ks, cur = collections.OrderedDict(), None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            ks[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(.*?);", line)
        if m and cur:
            ks[cur].append(m.group(1).strip())
    return ks


def main(old_dir, new_dir, renames=()):
    for name in sorted(f for f in os.listdir(new_dir) if f.endswith(".o")):
        old = kernels(os.path.join(old_dir, name)) if os.path.exists(os.path.join(old_dir, name)) else {}
        for a, b in renames:
            old = type(old)((k.replace(a, b), v) for k, v in old.items())
        new = kernels(os.path.join(new_dir, name))
        print("%s: %d kernels in the parent's build, %d in this one" % (name, len(old), len(new)))
        for k in list(old) + [k for k in new if k not in old]:
            if k not in new:
                print("  removed   %5d instr  %s" % (len(old[k]), k[:150]))
            elif k not in old:
                print("  new       %5d instr  %s" % (len(new[k]), k[:150]))
            elif old[k] == new[k]:
                print("  identical %5d instr  %s" % (len(new[k]), k[:150]))
            else:
                diff = sum(a != b for a, b in zip(old[k], new[k])) + abs(len(old[k]) - len(new[k]))
                print("  differs   %5d -> %5d instr (%d differ)  %s" % (len(old[k]), len(new[k]), diff, k[:150]))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2], [tuple(r.split("=", 1)) for r in sys.argv[3:]])
