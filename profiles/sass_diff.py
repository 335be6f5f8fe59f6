"""Per-kernel SASS comparison of two builds of libnfsp_b200.so (no GPU needed): instruction text and both encoding words,
addresses stripped.  Prints how many kernels are identical under the same name, and which differ, are new or are gone.

    python profiles/sass_diff.py PARENT_TREE/.../libnfsp_b200.so neural-ficititious-self-play-in-imperfect-information-games_b200/libnfsp_b200.so
"""
import re
import subprocess
import sys


def kernels(so):
    """{mangled kernel name: [(instruction, encoding word 1, encoding word 2), ...]} of the library's SASS."""
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    cur, d = None, {}
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            d[cur] = []
            continue
        if cur is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*/\*\s*(0x[0-9a-f]+)\s*\*/", line)
        if m:
            d[cur].append((m.group(1), m.group(2)))
            continue
        m = re.match(r"\s*/\*\s*(0x[0-9a-f]+)\s*\*/", line)   # the second encoding word, on a line of its own
        if m and d[cur]:
            d[cur][-1] = d[cur][-1] + (m.group(1),)
    return d


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    print("parent %d kernels, new %d" % (len(a), len(b)))
    print("identical under the same name: %d" % sum(1 for k in a if k in b and a[k] == b[k]))
    for k in a:
        if k not in b:
            print("GONE     ", k)
        elif a[k] != b[k]:
            print("DIFFERS  ", k, len(a[k]), "->", len(b[k]))
    for k in b:
        if k not in a:
            print("NEW      ", k, "(%d instructions)" % len(b[k]))


if __name__ == "__main__":
    main()
