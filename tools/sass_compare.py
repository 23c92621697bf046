"""Compares the SASS of kernels in two object files (e.g. a parent build and this tree's build of kernels_pre.cu.o), with
kernel names demangled and matched by a pattern per side, so a kernel that became a template instantiation can be compared with
its former self.  Instruction addresses are dropped; everything else (opcodes, registers, constant-bank offsets) must match.

    python tools/sass_compare.py OLD.o NEW.o "k_letterbox(=k_letterbox(" "k_warp_affine<(bool)0>=k_warp_affine<(bool)0, (bool)0>"

Prints per pair the instruction counts and the number of differing instructions (the first few shown); exit status 1 when any
pair differs.  Runs on the CPU (cuobjdump, cu++filt from the CUDA toolkit)."""
from __future__ import annotations

import os
import re
import subprocess
import sys

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def kernels(obj: str) -> dict:
    out = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", obj], capture_output=True, text=True, check=True).stdout
    ks, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = subprocess.run([os.path.join(CUDA, "bin", "cu++filt"), m.group(1)], capture_output=True, text=True).stdout.strip()
            ks[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            ks[cur].append(re.sub(r"/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip())
    return ks


def main() -> int:
    if len(sys.argv) < 4:
        print(__doc__)
        return 2
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    bad = 0
    for pair in sys.argv[3:]:
        pa, pb = pair.split("=")
        ka, kb = [k for k in a if pa in k], [k for k in b if pb in k]
        if len(ka) != 1 or len(kb) != 1:
            print("pattern %r / %r matches %s / %s" % (pa, pb, ka, kb))
            return 2
        A, B = a[ka[0]], b[kb[0]]
        diff = [(i, x, y) for i, (x, y) in enumerate(zip(A, B)) if x != y]
        n = len(diff) + abs(len(A) - len(B))
        bad += n > 0
        print("%s  vs  %s: %d / %d instructions, %d differ" % (ka[0], kb[0], len(A), len(B), n))
        for d in diff[:8]:
            print("    %d: %s  |  %s" % d)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
