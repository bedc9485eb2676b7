"""Kernel-by-kernel SASS comparison of two builds of the library (developer aid).

Usage: python scripts/sass_compare.py old.so new.so
Dumps both with `cuobjdump -sass`, strips addresses and symbol operands, and reports for every kernel of the OLD library whether
the new one holds the same instruction sequence. Names are matched after folding a bool template argument into the int of the
same value (`Lb0E` -> `Li0E`), so that a bool parameter widened to an int mode keeps its kernels paired, and after dropping a
trailing seventh template argument `false` of k_pairs, so that k_pairs<..., 32, false> pairs with k_pairs<..., 32>."""
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def kernels(path):
    text = subprocess.run([CUOBJDUMP, "-sass", path], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and name:
            out[name].append(re.sub(r"\b_Z\w+", "SYM", m.group(1)))
    return out


def key(name):
    name = re.sub(r"(7k_pairsI(?:L[ib]\d+E){6})Lb0EE", r"\1E", name)
    return re.sub(r"Lb([01])E", r"Li\1E", name)


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    new_by_key = {key(n): body for n, body in new.items()}
    same = 0
    for n, body in sorted(old.items()):
        other = new_by_key.get(key(n))
        if other is None:
            print("missing  ", n)
        elif other != body:
            print("different", n, len(body), len(other))
        else:
            same += 1
    added = sorted(set(new_by_key) - {key(n) for n in old})
    print("%d of %d kernels of the old library identical (%d instructions); %d kernels only in the new one:" %
          (same, len(old), sum(len(b) for b in old.values()), len(added)))
    for n in added:
        print("  ", n)
    return 0 if same == len(old) else 1


if __name__ == "__main__":
    sys.exit(main())
