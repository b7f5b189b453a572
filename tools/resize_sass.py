"""SASS of the resize front end (csrc/resize.cu): per kernel instantiation, its instructions (cuobjdump -sass) and what
ptxas reports (registers, spill bytes).

    python tools/resize_sass.py                 # the working tree: registers and spills per instantiation
    python tools/resize_sass.py --rev HEAD~1    # and whether every instantiation that exists at REV is instruction for
                                                # instruction the same in the working tree (exit 1 if not)

Names are compared with a trailing `false` template argument removed: a kernel template that gains a defaulted bool
parameter keeps its old instantiations under that name.  Compiles only (nvcc cross-compiles without a GPU)."""
import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "yolo-compression-and-deployment-in-fpga_b200"
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def nvcc():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if p and os.path.exists(p):
            return p
    return "nvcc"


def cuobjdump():
    p = os.path.join(os.path.dirname(nvcc()), "cuobjdump")
    return p if os.path.exists(p) else "cuobjdump"


def canonical(name):
    """A mangled resize_u8c3_kernel name without a trailing `false` (Lb0E) template argument."""
    return re.sub(r"ELb0EEEv", "EEEv", name)


def compile_resize(root):
    """{canonical name: (sass text, registers, spill store bytes)} of <root>/<PKG>/csrc/resize.cu."""
    with tempfile.TemporaryDirectory() as td:
        cubin = os.path.join(td, "resize.cubin")
        r = subprocess.run([nvcc()] + FLAGS + ["-cubin", "-o", cubin, os.path.join(root, PKG, "csrc", "resize.cu")],
                           capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed")
        info, cur = {}, None
        for line in r.stderr.splitlines():
            m = re.search(r"Compiling entry function '(\w+)'", line)
            if m:
                cur = canonical(m.group(1))
                info[cur] = [0, 0]
            m = re.search(r"(\d+) bytes spill stores", line)
            if m and cur:
                info[cur][1] = int(m.group(1))
            m = re.search(r"Used (\d+) registers", line)
            if m and cur:
                info[cur][0] = int(m.group(1))
        sass = subprocess.run([cuobjdump(), "-sass", cubin], capture_output=True, text=True, check=True).stdout
    out = {}
    for block in sass.split("Function : ")[1:]:
        name, _, body = block.partition("\n")
        name = canonical(name.strip())
        lines = [ln.strip() for ln in body.splitlines() if ln.strip() and not ln.strip().startswith(".")]
        out[name] = ("\n".join(lines), info[name][0], info[name][1])
    return out


def tree_at(rev, td):
    """The csrc and include directories of git revision rev, extracted under td."""
    arch = subprocess.run(["git", "-C", ROOT, "archive", rev, PKG + "/csrc", "include"], capture_output=True, check=True).stdout
    subprocess.run(["tar", "x", "-C", td], input=arch, check=True)
    return td


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rev", help="git revision whose instantiations must be unchanged")
    a = ap.parse_args()
    now = compile_resize(ROOT)
    for name, (_, regs, spill) in sorted(now.items()):
        print("%-70s %3d registers %4d bytes spilled" % (name, regs, spill))
    if not a.rev:
        return 0
    with tempfile.TemporaryDirectory() as td:
        old = compile_resize(tree_at(a.rev, td))
    same = [n for n in old if n in now and now[n][0] == old[n][0]]
    print("%d of %d instantiations of %s compile to the same SASS; %d new" % (len(same), len(old), a.rev, len(set(now) - set(old))))
    for n in sorted(set(old) - set(same)):
        print("DIFFERENT OR MISSING:", n)
    return 0 if len(same) == len(old) else 1


if __name__ == "__main__":
    sys.exit(main())
