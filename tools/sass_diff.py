"""Diff the SASS of every kernel of a base revision against the working tree's build of the same kernel (sm_100a, the library's
flags).  Kernels only the working tree has are listed as new, not compared.  Runs on the CPU: nvcc and cuobjdump need no GPU.

    python3 tools/sass_diff.py [--base HEAD] [--sources kernels.cu corr.cu]

Exit status 0 when every kernel of the base build has byte-identical SASS in the working tree's build."""
import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def sass(tree, source, out):
    csrc = os.path.join(tree, "digital-filtering_b200", "csrc")
    subprocess.run([NVCC, *FLAGS, "-I", os.path.join(tree, "include"), "-cubin", os.path.join(csrc, source), "-o", out], check=True, cwd=csrc)
    text = subprocess.run([CUOBJDUMP, "-sass", out], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))   # the anonymous namespace is hashed with the path
            funcs[name] = []
        elif name and line.strip():
            funcs[name].append(line.strip())
    return funcs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--base", default="HEAD")
    ap.add_argument("--sources", nargs="+", default=["kernels.cu", "corr.cu"])
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        base = os.path.join(tmp, "base")
        os.makedirs(base)
        archive = subprocess.run(["git", "-C", ROOT, "archive", a.base, "digital-filtering_b200/csrc", "include"], check=True,
                                 capture_output=True).stdout
        subprocess.run(["tar", "x", "-C", base], input=archive, check=True)
        same = differ = new = 0
        for src in a.sources:
            old = sass(base, src, os.path.join(tmp, "base_" + src + ".cubin"))
            cur = sass(ROOT, src, os.path.join(tmp, "cur_" + src + ".cubin"))
            for name in sorted(old):
                if name not in cur:
                    print(f"MISSING {src}: {name}")
                    differ += 1
                elif cur[name] != old[name]:
                    print(f"DIFFERS {src}: {name} ({len(old[name])} -> {len(cur[name])} lines)")
                    differ += 1
                else:
                    same += 1
            for name in sorted(set(cur) - set(old)):
                print(f"new     {src}: {name}")
                new += 1
        print(f"{same} kernels of {a.base} identical, {differ} differ or are missing, {new} new")
        return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
