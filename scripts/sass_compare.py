"""Compares the sm_100a SASS of two builds of the library, kernel by kernel: every kernel of the first build must have
byte-identical instructions in the second.  Kernels only the second build has are listed.
Needs cuobjdump, no GPU.
usage: python scripts/sass_compare.py old.so new.so"""
import re
import subprocess
import sys


def kernels(lib):
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,5}\*/\s+(.*?;)\s+/\* (0x[0-9a-f]+) \*/", line)   # instruction + first encoding word
        if m and cur is not None:
            cur.append(m.group(1) + " " + m.group(2))
        m = re.match(r"\s+/\* (0x[0-9a-f]+) \*/\s*$", line)                             # second encoding word
        if m and cur is not None:
            cur.append(m.group(1))
    return out


def main(old, new):
    a, b = kernels(old), kernels(new)
    changed = [k for k in a if k not in b or a[k] != b[k]]
    for k in sorted(a):
        print(("unchanged " if k not in changed else "CHANGED   ") + k)
    for k in sorted(set(b) - set(a)):
        print("new       " + k)
    print(f"{len(a) - len(changed)} of {len(a)} kernels unchanged, {len(set(b) - set(a))} new")
    return 1 if changed else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
