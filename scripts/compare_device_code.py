#!/usr/bin/env python
"""Compare the device code of two builds: for every object present in both directories (prost_b200/lib/obj of two
checkouts), `cuobjdump -sass` and `cuobjdump -res-usage` must agree.  A change that touches host code only leaves
them identical.  Two things differ between builds of the same device code and are normalised away: the
`identifier =` lines, which hold the source path, and the 8-hex-digit hash in anonymous-namespace names, which
changes with the file's contents.

  python scripts/compare_device_code.py OLD_OBJ_DIR NEW_OBJ_DIR
"""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
ANON = re.compile(r"_GLOBAL__N__[0-9a-f]{8}_")


def dump(path, flag):
    out = subprocess.run([CUOBJDUMP, flag, path], check=True, capture_output=True, text=True).stdout
    return [ANON.sub("_GLOBAL__N__X_", line) for line in out.splitlines() if "identifier =" not in line]


def main(old_dir, new_dir):
    old, new = set(os.listdir(old_dir)), set(os.listdir(new_dir))
    objs = sorted(n for n in old & new if n.endswith(".o"))
    bad = sorted(old ^ new)
    if bad:
        print("only in one build:", " ".join(bad))
    for name in objs:
        sass = [dump(os.path.join(d, name), "-sass") for d in (old_dir, new_dir)]
        res = [dump(os.path.join(d, name), "-res-usage") for d in (old_dir, new_dir)]
        kernels = sum(line.lstrip().startswith("Function :") for line in sass[1])
        same = sass[0] == sass[1] and res[0] == res[1]
        print(f"{name:24s} {kernels:4d} kernels  {'identical' if same else 'DIFFERENT'}")
        if not same:
            bad.append(name)
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
