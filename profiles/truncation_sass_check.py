"""Check that the truncation flag left the keep-mode step kernels' machine code alone.

Builds the given parent commit (in a temporary git worktree) and this working tree with walker_gym_b200/build.py, both
into temporary directories (nothing in the tree is written), and compares `cuobjdump -sass` of every kernel of the
given translation units, with constant-bank operands normalised: appending
`truncated` to StepArgs moves no existing parameter, but it may move the offsets of the constants that follow the
kernel parameters.  Prints, per kernel, the instruction counts, the register counts and whether the normalised
instruction sequences are identical.

    python profiles/truncation_sass_check.py PARENT_REV [unit ...]
(default units: wg_inst_balance_packed wg_inst_balance wg_inst_units wg_inst_units_link).  Exit status 0 when every
kernel is unchanged.
"""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(tree, out):
    """Object files of `tree` in `out` (build.py with WG_OBJ_DIR / WG_LIB_OUT pointing there)."""
    env = dict(os.environ, WG_OBJ_DIR=os.path.join(out, "obj"), WG_LIB_OUT=os.path.join(out, "lib.so"))
    subprocess.run([sys.executable, os.path.join(tree, "walker_gym_b200", "build.py"), "--force"], env=env, check=True,
                   stdout=subprocess.DEVNULL)
    return env["WG_OBJ_DIR"]


def kernels(obj):
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    res = subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True, check=True).stdout
    regs = {}
    name = None
    for line in res.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
        m = re.search(r"REG:(\d+)", line)
        if m and name:
            regs[name] = int(m.group(1))
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if cur and m:
            ins = re.sub(r"c\[0x[0-9a-f]+\]\[0x[0-9a-f]+\]", "c[B][O]", m.group(1))
            out[cur].append(ins)
    return {k: (v, regs.get(k)) for k, v in out.items()}


def main():
    rev = sys.argv[1]
    units = sys.argv[2:] or ["wg_inst_balance_packed", "wg_inst_balance", "wg_inst_units", "wg_inst_units_link"]
    with tempfile.TemporaryDirectory() as tmp:
        wt = os.path.join(tmp, "parent")
        subprocess.run(["git", "-C", ROOT, "worktree", "add", "--detach", "-q", wt, rev], check=True)
        try:
            old_dir = build(wt, os.path.join(tmp, "old"))
        finally:
            subprocess.run(["git", "-C", ROOT, "worktree", "remove", "--force", wt], check=False)
        new_dir = build(ROOT, os.path.join(tmp, "new"))
        return compare(old_dir, new_dir, units)


def compare(old_dir, new_dir, units):
    same_all = True
    for u in units:
        a, b = kernels(f"{old_dir}/{u}.o"), kernels(f"{new_dir}/{u}.o")
        for k in sorted(set(a) | set(b)):
            if k not in a or k not in b:
                print(f"{u}: {k} only in {'parent' if k in a else 'this tree'}")
                same_all = False
                continue
            (ia, ra), (ib, rb) = a[k], b[k]
            same = ia == ib
            same_all &= same and ra == rb
            print(f"{u}: {'same' if same else 'DIFFERENT'} instr {len(ia)} -> {len(ib)} regs {ra} -> {rb}  {k[:110]}")
    return 0 if same_all else 1


if __name__ == "__main__":
    sys.exit(main())
