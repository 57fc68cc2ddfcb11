"""Registers, shared memory and spills of every kernel of the convolution sources, as ptxas reports them.

    python tools/kernel_resources.py [--root TREE] [files ...]     (default: conv_tc.cu conv_simt.cu)

Compiles each source for sm_100a with the library's flags (``mm2d3d_b200/build.py``) plus ``-Xptxas -v`` into a
temporary directory and prints one line per kernel instantiation, demangled.  No GPU needed.  Run it on two trees to
compare them (``--root`` = a checkout of the parent commit)."""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def usage(root, name):
    sys.path.insert(0, ROOT)
    from mm2d3d_b200.build import NVCC_FLAGS, _nvcc
    src = os.path.join(root, "mm2d3d_b200", "csrc", name)
    flags = [f if not f.endswith("/include") else os.path.join(root, "include") for f in NVCC_FLAGS]
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([_nvcc(), *flags, "-Xptxas", "-v", "-c", src, "-o", os.path.join(tmp, "k.o")],
                           capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(r.stderr)
    rows, fn, spill = [], None, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            fn = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            spill = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and fn:
            smem = re.search(r"(\d+) bytes smem", line)
            rows.append((fn, int(m.group(1)), int(smem.group(1)) if smem else 0, spill))
            fn = None
    names = subprocess.run(["c++filt"], input="\n".join(r[0] for r in rows), capture_output=True, text=True).stdout.split("\n")
    return [(n.strip(), *r[1:]) for n, r in zip(names, rows)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("files", nargs="*", default=["conv_tc.cu", "conv_simt.cu"])
    a = ap.parse_args()
    for f in a.files:
        for name, regs, smem, spill in usage(a.root, f):
            print(f"{f:14s} regs {regs:4d}  smem {smem:6d}  spill st/ld {spill[0]}/{spill[1]}  {name}")


if __name__ == "__main__":
    main()
