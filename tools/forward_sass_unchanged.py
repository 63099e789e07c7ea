"""Check that the forward k-NN kernels compile to the same machine code as at another commit (no GPU needed).

    python tools/forward_sass_unchanged.py [--base REV]      # default REV: HEAD~1

Compiles hm_tc.cu, hm_popc.cu and hm_small.cu of the working tree and of REV (sources taken with `git show`) to sm_100a
cubins with the flags of slam_experiments_b200/build.py plus `-Xptxas -v`, then compares, per file, the SASS of every
kernel (`cuobjdump -sass` with instruction addresses and the path hash of anonymous namespaces stripped) and the ptxas register / stack / spill
lines.  Exit status 0 iff everything is identical.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FILES = ("hm_tc.cu", "hm_popc.cu", "hm_small.cu")
TREE = ("include/hm_matcher.h", "slam_experiments_b200/csrc")


def export_rev(rev, dst):
    for path in TREE:
        names = subprocess.run(["git", "ls-tree", "-r", "--name-only", rev, path], cwd=ROOT, check=True,
                               capture_output=True, text=True).stdout.split()
        for n in names:
            os.makedirs(os.path.join(dst, os.path.dirname(n)), exist_ok=True)
            with open(os.path.join(dst, n), "wb") as f:
                f.write(subprocess.run(["git", "show", f"{rev}:{n}"], cwd=ROOT, check=True, capture_output=True).stdout)


def compile_one(root, name, out_dir):
    from slam_experiments_b200.build import nvcc_path
    cubin = os.path.join(out_dir, name + ".cubin")
    r = subprocess.run([nvcc_path(), "-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xptxas", "-v", "-I", os.path.join(root, "include"), "-I",
                        os.path.join(root, "slam_experiments_b200", "csrc"), "-cubin", "-o", cubin,
                        os.path.join(root, "slam_experiments_b200", "csrc", name)],
                       check=True, capture_output=True, text=True)
    ptxas = [l.strip() for l in r.stderr.splitlines() if re.search(r"registers|stack frame|spill", l)]
    cuobjdump = os.path.join(os.path.dirname(nvcc_path()), "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", cubin], check=True, capture_output=True, text=True).stdout
    # instruction addresses go; so does the hash of the source path in anonymous-namespace names
    sass = [re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", re.sub(r"/\*[0-9a-f]{4,}\*/", "", l)).strip()
            for l in sass.splitlines()]
    return [l for l in sass if l], ptxas


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default="HEAD~1")
    args = ap.parse_args()
    same = True
    with tempfile.TemporaryDirectory() as tmp:
        base_root = os.path.join(tmp, "base")
        export_rev(args.base, base_root)
        for name in FILES:
            a_sass, a_ptx = compile_one(base_root, name, tmp)
            b_sass, b_ptx = compile_one(ROOT, name, tmp)
            kernels = sum(1 for l in b_sass if l.startswith("Function :"))
            ok = a_sass == b_sass and a_ptx == b_ptx
            same &= ok
            print(f"{name}: {kernels} kernels, SASS {'identical' if a_sass == b_sass else 'DIFFERS'}, "
                  f"ptxas figures {'identical' if a_ptx == b_ptx else 'DIFFER'} ({len(b_ptx)} lines)")
    print("forward kernels unchanged" if same else "forward kernels CHANGED")
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
