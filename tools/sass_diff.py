"""Which kernels of two builds of libf3ps.so compile to different SASS.

  cuobjdump -sass old/libf3ps.so > old.sass; cuobjdump -sass libf3ps.so > new.sass
  python tools/sass_diff.py old.sass new.sass

Kernels are matched by mangled name with the per-file hash of anonymous namespaces removed; instruction addresses are
ignored.  Prints the kernels only one build has and those whose instructions differ."""
import re
import sys


def kernels(path):
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))
            out[cur] = []
        elif cur:
            ins = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()
            if ins:
                out[cur].append(ins)
    return out


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    print("kernels: %d before, %d after" % (len(a), len(b)))
    print("only before:", sorted(set(a) - set(b)))
    print("only after:", sorted(set(b) - set(a)))
    print("changed:", sorted(k for k in a if k in b and a[k] != b[k]))
    print("unchanged: %d" % sum(1 for k in a if k in b and a[k] == b[k]))


if __name__ == "__main__":
    main()
