"""Kernel-by-kernel comparison of the SASS of two builds of libicp_gpu.so (cuobjdump -sass): which kernels compile to the same
instructions.  Anonymous-namespace hashes (they depend on the source path) and the address comments are normalised away; cuobjdump's
section markers are not instructions and are skipped.
Usage: python profiles/compare_sass.py parent.so this.so [exclude-substring ...]"""
import re
import subprocess
import sys


def kernels(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], stdout=subprocess.PIPE, text=True, check=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))
            d[cur] = []
            continue
        if cur is None:
            continue
        line = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()
        if ";" in line:                                   # an instruction (its encoding lines and markers carry none)
            d[cur].append(line)
    return d


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    skip = sys.argv[3:]
    same, diff = [], []
    for k in sorted(a):
        if any(s in k for s in skip):
            continue
        (same if k in b and a[k] == b[k] else diff).append(k)
    new = sorted(k for k in b if k not in a)
    print(f"kernels compared: {len(same) + len(diff)} (excluded: {', '.join(skip) or 'none'})")
    print(f"identical instructions: {len(same)}")
    print(f"different: {len(diff)}" + "".join(f"\n  {k}" for k in diff))
    print(f"only in the second build: {len(new)}" + "".join(f"\n  {k}" for k in new))


if __name__ == "__main__":
    main()
