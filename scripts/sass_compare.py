"""Compares the sm_100a SASS of two builds of the library, kernel by kernel: every kernel of the first build must have
byte-identical instructions in the second.  A kernel that gained a trailing template parameter with the value false (the
SIZED flag of the kernels that take per-image extents, e.g. center_kernel<false, 0, true> ->
center_kernel<false, 0, true, false>) is matched to its old name.  Kernels only the second build has are listed.
Needs cuobjdump and cu++filt, no GPU.
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


def demangle(names):
    """mangled name -> name with its template arguments, without return type and parameter list"""
    out = subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    plain = [v.replace("void ", "", 1) for v in out.splitlines()]
    return {k: v[: v.index(">(") + 1] if ">(" in v else v[: v.index("(")] for k, v in zip(names, plain)}


def main(old, new):
    a, b = kernels(old), kernels(new)
    plain_a, plain_b = demangle(list(a)), demangle(list(b))
    by_plain = {v: k for k, v in plain_a.items()}
    for k in list(b):
        if k in a:
            continue
        plain = plain_b[k]
        for tail, repl in ((", (bool)0>", ">"), ("<(bool)0>", "")):   # cu++filt spells false as (bool)0
            if plain.endswith(tail):
                plain = plain[: -len(tail)] + repl
                break
        old_name = by_plain.get(plain)
        if old_name is not None and old_name not in b:
            b[old_name] = b.pop(k)
    changed = [k for k in a if k not in b or a[k] != b[k]]
    for k in sorted(a):
        print(("unchanged " if k not in changed else "CHANGED   ") + k)
    for k in sorted(set(b) - set(a)):
        print("new       " + k)
    print(f"{len(a) - len(changed)} of {len(a)} kernels unchanged, {len(set(b) - set(a))} new")
    return 1 if changed else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
