"""Compare the machine code of the step kernels between two trees: the parent commit and the working tree.

    python tools/sass_diff.py [--base REV] [--keep DIR]

Both trees are compiled for sm_100a with the flags of ppo-2dgrid_b200/build.py into a temporary directory (no GPU
needed; about 16 s each on 8 cores), `cuobjdump -sass` is split per function, and every function present in both
libraries is compared instruction by instruction after dropping the /*addr*/ columns and normalising the
`_GLOBAL__N__<hash>` / `_INTERNAL_<hash>` names, which depend on the build path.

The one difference accepted is a kernel-parameter offset: a field appended to EnvParams moves the parameter that
follows it (`c[0x0][0x4d0]` -> `c[0x0][0x4d8]`).  A line pair passes when its only difference is constant-bank-0
offsets that all moved by the same amount; the tool prints which offsets moved.  Exit status 1 if any function
present in both differs in any other way.

--base defaults to HEAD when the CUDA sources differ from HEAD, else HEAD~1 (the parent of the checked-out commit).
"""
from __future__ import annotations

import argparse
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ppo-2dgrid_b200")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
SOURCES = ("ppo-2dgrid_b200/csrc", "include")

_ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")
_HASH = re.compile(r"(_GLOBAL__N__|_INTERNAL_)[0-9a-f]+(_[0-9]+_\w+?_cu_[0-9a-f]+)?")
_CBANK = re.compile(r"c\[0x0\]\[(0x[0-9a-f]+)\]")


def _build_flags():
    sys.path.insert(0, PKG)
    import build  # ppo-2dgrid_b200/build.py
    return [f for f in build.FLAGS if not f.startswith("-I")]


def _compile(tree, out):
    csrc = os.path.join(tree, "ppo-2dgrid_b200", "csrc")
    srcs = sorted(os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cu"))
    cmd = [os.path.join(CUDA, "bin", "nvcc")] + _build_flags() + [
        "-I" + os.path.join(tree, "include"), "-I" + csrc, "-o", out] + srcs
    subprocess.check_call(cmd)


def _functions(so):
    text = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", so], capture_output=True, text=True,
                          check=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = _HASH.sub(r"\1", m.group(1))
            funcs[cur] = []
            continue
        if cur is not None and _ADDR.search(line):
            ins = _ADDR.sub("", line).split(";")[0].strip()
            funcs[cur].append(_HASH.sub(r"\1", ins))
    return funcs


def _demangle(name):
    return subprocess.run(["c++filt"], input=name, capture_output=True, text=True).stdout.strip()


def _compare(old, new):
    """None when identical, a set of (old, new) parameter offsets when only those moved (by one common amount),
    else a string describing the first other difference."""
    if len(old) != len(new):
        return f"{len(old)} vs {len(new)} instructions"
    moved = set()
    for i, (a, b) in enumerate(zip(old, new)):
        if a == b:
            continue
        if _CBANK.sub("c[]", a) != _CBANK.sub("c[]", b):
            return f"instruction {i}: {a!r} vs {b!r}"
        for x, y in zip(_CBANK.findall(a), _CBANK.findall(b)):
            if x != y:
                moved.add((int(x, 16), int(y, 16)))
    if not moved:
        return None
    if len({y - x for x, y in moved}) != 1:
        return f"parameter offsets moved by different amounts: {sorted(moved)}"
    return moved


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--base", default=None, help="git revision to compare against")
    ap.add_argument("--keep", default=None, help="directory to keep the two libraries in")
    args = ap.parse_args()
    base = args.base
    if base is None:
        dirty = subprocess.run(["git", "-C", ROOT, "diff", "--quiet", "HEAD", "--", *SOURCES]).returncode != 0
        base = "HEAD" if dirty else "HEAD~1"
    rev = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", base], capture_output=True, text=True,
                         check=True).stdout.strip()
    tmp = tempfile.mkdtemp(prefix="sass_diff_")
    try:
        old_tree, new_tree = os.path.join(tmp, "base"), os.path.join(tmp, "tree")
        os.makedirs(old_tree)
        archive = subprocess.run(["git", "-C", ROOT, "archive", base, *SOURCES], capture_output=True, check=True).stdout
        subprocess.run(["tar", "-x", "-C", old_tree], input=archive, check=True)
        for d in SOURCES:
            shutil.copytree(os.path.join(ROOT, d), os.path.join(new_tree, d))
        old_so, new_so = os.path.join(tmp, "base.so"), os.path.join(tmp, "tree.so")
        _compile(old_tree, old_so)
        _compile(new_tree, new_so)
        old, new = _functions(old_so), _functions(new_so)
        if args.keep:
            os.makedirs(args.keep, exist_ok=True)
            shutil.copy(old_so, os.path.join(args.keep, "base.so"))
            shutil.copy(new_so, os.path.join(args.keep, "tree.so"))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    common = [k for k in old if k in new]
    same = [k for k in common if old[k] == new[k]]
    shifted, failed = [], []
    for k in common:
        if k in same:
            continue
        r = _compare(old[k], new[k])
        (shifted if isinstance(r, set) else failed).append((k, r))
    print(f"base {rev}: {len(old)} functions; working tree: {len(new)} functions ({len(new) - len(common)} new)")
    print(f"  identical: {len(same)}")
    print(f"  identical up to the parameter offset after EnvParams: {len(shifted)}")
    for k, moved in shifted:
        print(f"    {_demangle(k)}: " + ", ".join(f"c[0x0][{x:#x}] -> {y:#x}" for x, y in sorted(moved)))
    print(f"  different: {len(failed)}")
    for k, why in failed:
        print(f"    {_demangle(k)}: {why}")
    missing = [k for k in old if k not in new]
    if missing:
        print(f"  absent from the working tree: {len(missing)}")
        for k in missing:
            print(f"    {_demangle(k)}")
    return 1 if failed or missing else 0


if __name__ == "__main__":
    sys.exit(main())
