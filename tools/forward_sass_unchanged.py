"""Check that the forward k-NN kernels compile to the same machine code as at another commit (no GPU needed).

    python tools/forward_sass_unchanged.py [--base REV]      # default REV: HEAD~1

Compiles hm_tc.cu, hm_popc.cu and hm_small.cu of the working tree and of REV (sources taken with `git show`) to sm_100a
cubins with the flags of slam_experiments_b200/build.py plus `-Xptxas -v`, then compares, per kernel, the SASS
(`cuobjdump -sass` with instruction addresses and the path hash of anonymous namespaces stripped) and the ptxas register /
stack / spill lines.  Every kernel that exists at REV must be identical; kernels that REV does not have are listed
separately, with their ptxas figures.  Exit status 0 iff every kernel of REV is unchanged and still present.
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


def _anon(s):
    """the hash of the source path in anonymous-namespace names goes"""
    return re.sub(r"_GLOBAL__N__[0-9a-f]+_[0-9a-z_]*?_cu_[0-9a-f]+", "_GLOBAL__N__", s)


def compile_one(root, name, out_dir):
    """-> ({kernel: [SASS lines]}, {kernel: [ptxas figure lines]})"""
    from slam_experiments_b200.build import nvcc_path
    cubin = os.path.join(out_dir, name + ".cubin")
    r = subprocess.run([nvcc_path(), "-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xptxas", "-v", "-I", os.path.join(root, "include"), "-I",
                        os.path.join(root, "slam_experiments_b200", "csrc"), "-cubin", "-o", cubin,
                        os.path.join(root, "slam_experiments_b200", "csrc", name)],
                       check=True, capture_output=True, text=True)
    ptxas, cur = {}, None
    for l in r.stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?([\w$]+)'?", l)
        if m:
            cur = _anon(m.group(1))
        elif cur and re.search(r"registers|stack frame|spill", l):
            ptxas.setdefault(cur, []).append(re.sub(r"^ptxas info\s*:\s*", "", l.strip()))
    cuobjdump = os.path.join(os.path.dirname(nvcc_path()), "cuobjdump")
    sass, cur = {}, None
    for l in subprocess.run([cuobjdump, "-sass", cubin], check=True, capture_output=True, text=True).stdout.splitlines():
        l = _anon(re.sub(r"/\*[0-9a-f]{4,}\*/", "", l)).strip()
        m = re.match(r"Function : (\S+)", l)
        if m:
            cur = m.group(1)
            sass[cur] = []
        elif l and cur:
            sass[cur].append(l)
    return sass, ptxas


def short(kernel):
    m = re.search(r"(hm_\w+?_kernel)", kernel)
    return m.group(1) if m else kernel


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
            n_same = 0
            for k in sorted(a_sass):
                s_ok = b_sass.get(k) == a_sass[k]
                p_ok = b_ptx.get(k) == a_ptx.get(k)
                if k not in b_sass:
                    print(f"  {name}: {short(k)} MISSING")
                elif not (s_ok and p_ok):
                    print(f"  {name}: {short(k)} SASS {'identical' if s_ok else 'DIFFERS'}, "
                          f"ptxas figures {'identical' if p_ok else 'DIFFER'}")
                n_same += s_ok and p_ok
                same &= s_ok and p_ok
            print(f"{name}: {n_same} of {len(a_sass)} kernels of {args.base} identical (SASS and ptxas figures)")
            for k in sorted(set(b_sass) - set(a_sass)):
                print(f"  new: {short(k)}: {'; '.join(b_ptx.get(k, []))}")
    print("forward kernels unchanged" if same else "forward kernels CHANGED")
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
