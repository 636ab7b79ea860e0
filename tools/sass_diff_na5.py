"""Checks that the five-agent instantiations of the rollout kernels (policy.cu) are, instruction for instruction, the
kernels of a base revision that predates the agent-count template parameter.

    python tools/sass_diff_na5.py [--base REV]        (needs git and nvcc, no GPU)

REV defaults to the parent of the commit that replaced the single agent count `POL_NA = 5` by the template parameter,
found in the history of policy.cu, wherever HEAD is.

Both revisions' policy.cu are compiled to sm_100a cubins with the library's flags, `cuobjdump -sass` lists every
kernel, function names are stripped, and each base kernel is compared with the new kernel of the same name and NA = 5
(kernels without the parameter compare by name alone).  Exit status 0 and "identical" per kernel, else the first
differing lines."""
import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = "safe-marl_b200/csrc"
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false", "-cubin"]


def compile_cubin(tree, out):
    subprocess.run([os.path.join(CUDA, "bin", "nvcc"), *FLAGS, "-o", out, os.path.join(tree, CSRC, "policy.cu")], check=True)


def kernels(cubin):
    """{name: [instruction lines]}: name = the demangled kernel name with NA = 5 folded away, addresses kept (they are
    offsets from the kernel's start), the function name removed."""
    sass = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", cubin], check=True, capture_output=True, text=True).stdout
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            dem = subprocess.run([os.path.join(CUDA, "bin", "cu++filt")], input=m.group(1), capture_output=True, text=True).stdout
            name = re.search(r"::(k_\w+)(<\(int\)(\d)>)?", dem)
            cur = None if name.group(3) not in (None, "5") else name.group(1)
            if cur is not None:
                out[cur] = []
            continue
        if cur is not None and "/*" in line:
            out[cur].append(line.strip())
    return out


def default_base():
    """The parent of the last commit that changed how often `POL_NA = 5` occurs in policy.cu (the one that removed it)."""
    rev = subprocess.run(["git", "-C", ROOT, "log", "-1", "--format=%H", "-S", "POL_NA = 5", "--", f"{CSRC}/policy.cu"],
                         check=True, capture_output=True, text=True).stdout.strip()
    if not rev:
        sys.exit("no commit removes POL_NA = 5 from policy.cu in this history: pass --base")
    return rev + "~1"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default=None, help="the revision to compare with (default: see the module docstring)")
    args = ap.parse_args()
    args.base = args.base or default_base()
    print(f"base: {subprocess.run(['git', '-C', ROOT, 'rev-parse', '--short', args.base], capture_output=True, text=True).stdout.strip()}")
    with tempfile.TemporaryDirectory() as tmp:
        base = os.path.join(tmp, "base")
        os.makedirs(base)
        arch = subprocess.run(["git", "-C", ROOT, "archive", args.base, CSRC, "include"], check=True, capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", base], input=arch, check=True)
        compile_cubin(base, os.path.join(tmp, "base.cubin"))
        compile_cubin(ROOT, os.path.join(tmp, "new.cubin"))
        old, new = kernels(os.path.join(tmp, "base.cubin")), kernels(os.path.join(tmp, "new.cubin"))
    bad = 0
    for name in sorted(old):
        if name not in new:
            print(f"{name}: missing from the new build"); bad += 1; continue
        a, b = old[name], new[name]
        if a == b:
            print(f"{name}: identical ({len(a)} lines)")
            continue
        bad += 1
        i = next((k for k in range(min(len(a), len(b))) if a[k] != b[k]), min(len(a), len(b)))
        print(f"{name}: DIFFERS ({len(a)} vs {len(b)} lines) at line {i}:\n  base: {a[i] if i < len(a) else '-'}\n  new:  {b[i] if i < len(b) else '-'}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
