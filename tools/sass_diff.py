"""Compare the compiled kernels of two source trees function by function, without a GPU.

    python tools/sass_diff.py OLD_TREE NEW_TREE [fast_path.cu generic_path.cu ...]

Each source under ghost_b200/csrc is compiled to a cubin, in both trees with the flags of NEW_TREE's Makefile.  For every function the
tool prints whether its SASS is the same in both trees and, when it is not, the differing instructions; then
the ptxas resource lines (registers, shared memory, stack, spills) that differ.  Instructions are compared
without their addresses and encodings, branch targets are dropped (code removed before a branch moves them),
and constant-bank-3 operands are written as symbol + offset, so that a __constant__ array that moves without
changing what it holds does not count as a change.  A function that differs is listed with the instructions
only one side has, counted as multisets with register, predicate and barrier names and operand-reuse flags blanked out: ptxas
reallocates registers and reorders blocks throughout a function when one branch of it changes, which turns a
line diff into noise.  A function only one tree has is reported as `renamed OLD -> NEW` when its instructions
are identical to those of exactly one function only the other tree has, and their resource lines are compared
under that pairing.  A refactor that must leave the kernels alone should report every function `same` or `renamed`.
"""
import collections
import concurrent.futures
import os
import re
import subprocess
import sys
import tempfile


def nvcc_flags(tree):
    mk = open(os.path.join(tree, "ghost_b200", "csrc", "Makefile")).read()
    arch = re.search(r"^ARCH\s*:=\s*(.*)$", mk, re.M).group(1)
    return re.search(r"^NVCCFLAGS\s*:=\s*(.*)$", mk, re.M).group(1).replace("$(ARCH)", arch).split()


def build(tree, src, out, flags):
    nvcc = os.environ.get("NVCC", "nvcc")
    r = subprocess.run([nvcc] + flags + ["-cubin", os.path.join(tree, "ghost_b200", "csrc", src), "-o", out],
                       capture_output=True, text=True)
    if r.returncode:
        sys.exit("%s: %s" % (src, r.stderr))
    return r.stderr                                    # -Xptxas -v writes the resource lines here


def const3_symbols(cubin):
    elf = subprocess.run(["cuobjdump", "-elf", cubin], capture_output=True, text=True, check=True).stdout
    rows = [l.split() for l in elf.split(".section .symtab", 1)[1].splitlines()]
    rows = [r for r in rows if len(r) == 7]
    shndx = {r[6]: r[5] for r in rows}.get(".nv.constant3")
    return [(int(r[1], 16), int(r[2], 16), r[6]) for r in rows if r[5] == shndx and not r[6].startswith(".")]


def sass(cubin):
    syms = const3_symbols(cubin)

    def const3(m):
        a = int(m.group(1), 16)
        for lo, size, name in syms:
            if lo <= a < lo + size:
                return "c[0x3][%s+%#x]" % (name, a - lo)
        return m.group(0)

    funcs, cur = {}, None
    for l in subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout.splitlines():
        m = re.search(r"Function : (\S+)", l)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(.*?)\s*;", l)
        if m and cur is not None:
            ins = re.sub(r"c\[0x3\]\[(0x[0-9a-f]+)\]", const3, m.group(1))
            ins = re.sub(r"^((?:@!?U?P\w+\s+)?(?:BRA|BSSY|CALL|BRX|JMP)\S*\s.*?)\s*0x[0-9a-f]+$", r"\1 <target>", ins)
            cur.append(ins)
    return funcs


def blank(ins):
    ins = re.sub(r"\bB\d+\b", "B", ins.replace(".reuse", ""))
    return re.sub(r"\bU?R\d+\b", "R", re.sub(r"\bU?P\d\b", "P", ins))


def resources(ptxas):
    res, cur = {}, None
    for l in ptxas.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", l)
        if m:
            cur = m.group(1)
        elif cur and re.search(r"Used \d+ registers|bytes stack frame", l):
            res[cur] = (res.get(cur, "") + " " + l.replace("ptxas info    :", "").strip()).strip()
    return res


def main():
    if len(sys.argv) < 3:
        sys.exit(__doc__)
    old, new = sys.argv[1], sys.argv[2]
    srcs = sys.argv[3:] or ["fast_path.cu", "generic_path.cu"]
    lines = int(os.environ.get("SASS_DIFF_LINES", "60"))
    flags = nvcc_flags(new)
    changed = 0
    with tempfile.TemporaryDirectory() as tmp, concurrent.futures.ThreadPoolExecutor(2) as pool:
        for src in srcs:
            cub = {s: os.path.join(tmp, "%s_%s.cubin" % (s, src)) for s in ("old", "new")}
            jobs = {s: pool.submit(build, t, src, cub[s], flags) for s, t in (("old", old), ("new", new))}
            ptx = {s: j.result() for s, j in jobs.items()}
            fo, fn = sass(cub["old"]), sass(cub["new"])
            print("==", src, "(%d functions old, %d new)" % (len(fo), len(fn)))
            # a function only one side has is a rename when exactly one function of the other side has its code
            by_code = collections.defaultdict(lambda: ([], []))
            for side, funcs, other in ((0, fo, fn), (1, fn, fo)):
                for f in funcs:
                    if f not in other:
                        by_code[tuple(funcs[f])][side].append(f)
            renamed = {a[0]: b[0] for a, b in by_code.values() if len(a) == 1 and len(b) == 1}
            for f in sorted(set(fo) | set(fn)):
                if f in renamed:
                    print("renamed   %s -> %s" % (f, renamed[f]))
                elif f in renamed.values():
                    continue
                elif f not in fo or f not in fn:
                    print("%-9s %s" % ("new only" if f in fn else "old only", f))
                    changed += 1
                elif fo[f] == fn[f]:
                    print("same      %s" % f)
                else:
                    a, b = collections.Counter(map(blank, fo[f])), collections.Counter(map(blank, fn[f]))
                    gone, came = a - b, b - a
                    print("differs   %s  (%d -> %d instructions; apart from register names -%d +%d)" % (
                        f, len(fo[f]), len(fn[f]), sum(gone.values()), sum(came.values())))
                    d = ["- %3d  %s" % (n, i) for i, n in gone.items()] + ["+ %3d  %s" % (n, i) for i, n in came.items()]
                    for l in d[:lines]:
                        print("    " + l)
                    changed += 1
            ro, rn = resources(ptx["old"]), resources(ptx["new"])
            rn.update({f: rn.pop(g) for f, g in renamed.items() if g in rn})       # compare renamed pairs
            diff = [f for f in sorted(set(ro) | set(rn)) if ro.get(f) != rn.get(f)]
            print("ptxas resources: %s" % ("identical for all %d functions" % len(rn) if not diff else "differ"))
            for f in diff:
                print("    %s\n      old: %s\n      new: %s" % (f, ro.get(f), rn.get(f)))
    return 1 if changed else 0


if __name__ == "__main__":
    sys.exit(main())
