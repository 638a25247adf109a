#!/usr/bin/env python
"""Kernel-by-kernel comparison of two builds of the library (python -m spalinalg_b200.build --force in each tree).

For every kernel of every object under <tree>/spalinalg_b200/build/ it compares
  * the `cuobjdump -sass` listing: instruction text and encodings, with the /*addr*/ column dropped and the
    anonymous-namespace prefix (_GLOBAL__N__<hash>_<n>_<file>_cu_<hash>, which follows the file's contents) removed;
  * registers, spills and static shared memory from the ptxas -v log (the profiles/ptxas_summary.py table).
A kernel is identical when its listing (instructions and encodings) and its resources are.  Prints the count of
identical kernels per object, then every changed kernel with its changed SASS instructions, its
registers before -> after, its spills and the CTAs per SM its registers allow (288- and 320-thread CTAs, 64 K
registers per SM, allocation in 256-register units per warp, capped by the CTAs __launch_bounds__ asks for).

Usage: python profiles/r4_sass_compare.py PARENT_TREE PR_TREE"""
import difflib
import glob
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
ANON = re.compile(r"(\d+)_GLOBAL__N__")


def strip_anon(text):
    """Drop every length-prefixed anonymous-namespace component of a mangled name."""
    out, pos = [], 0
    for m in ANON.finditer(text):
        if m.start() < pos:
            continue
        out.append(text[pos:m.start()])
        pos = m.start() + len(m.group(1)) + int(m.group(1))
    out.append(text[pos:])
    return "".join(out)


def demangle(name):
    d = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
    return re.sub(r"\(anonymous namespace\)::|spl::|^void ", "", d).split("(")[0]


NAMES = {}      # mangled name without the anonymous prefix -> demangled name


def sass(obj):
    """{mangled name without the anonymous prefix: [(instruction, encoding)]}: the instruction text with branch
    targets relative to the instruction (code that grows or shrinks elsewhere moves every absolute target), and the
    text and encoding words as listed, both without the /*addr*/ column"""
    text = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, cur, addr = {}, None, 0
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            key = strip_anon(m.group(1))
            if key not in NAMES:
                NAMES[key] = demangle(m.group(1))
            cur = funcs.setdefault(key, [])
            continue
        if cur is None or not line.strip() or ".headerflags" in line:
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s*(.*?)\s*(/\*.*\*/)\s*$", line)
        if m:
            addr = int(m.group(1), 16)
            ins = re.sub(r"(BRA|BSSY\S*|CALL\S*|SSY|PBK|BRX)(.*?)0x([0-9a-f]+)",
                         lambda b: f"{b.group(1)}{b.group(2)}.{(int(b.group(3), 16) - addr) // 16:+d}", m.group(2))
            cur.append((strip_anon(ins), strip_anon(m.group(2) + " " + m.group(3))))
        elif cur:                                   # second encoding word of the instruction above
            cur[-1] = (cur[-1][0], cur[-1][1] + " " + line.strip())
    return funcs


def resources(log):
    """{mangled name without the anonymous prefix: (registers, spill stores, spill loads, static smem)}"""
    res, name, spill = {}, None, (0, 0)
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = strip_anon(m.group(1))
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            spill = (int(m.group(1)), int(m.group(2)))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            smem = re.search(r"(\d+) bytes smem", line)
            res[name] = (int(m.group(1)), spill[0], spill[1], int(smem.group(1)) if smem else 0)
            name, spill = None, (0, 0)
    return res


def ctas_by_regs(regs, threads):
    per_warp = (regs * 32 + 255) // 256 * 256
    return 65536 // (per_warp * ((threads + 31) // 32))


def launch_shape(name):
    """(threads per CTA, __launch_bounds__ minimum CTAs per SM) of the stream and fused-gather kernels; other
    kernels: 256 threads, no cap"""
    if name.startswith("spmv_gather_fused_kernel"):
        return 320, 4
    if name.startswith("spmv_stream_kernel"):
        tight = name.split("<", 1)[1].split(", ")[3] == "true"      # <T, LPR, U, TIGHT, PAT, XG>
        return 288, 4 if tight else 3
    return 256, 64


def changed_lines(a, b):
    """instructions inserted, deleted or replaced between the two listings (text, relative branch targets)"""
    a, b = [i for i, _ in a], [i for i, _ in b]
    n = 0
    for tag, i1, i2, j1, j2 in difflib.SequenceMatcher(None, a, b, autojunk=False).get_opcodes():
        if tag != "equal":
            n += max(i2 - i1, j2 - j1)
    return n


def main(parent, pr):
    objs = sorted(os.path.basename(p) for p in glob.glob(os.path.join(pr, "spalinalg_b200", "build", "*.o")))
    changed = []
    for o in objs:
        pa, pb = (os.path.join(t, "spalinalg_b200", "build", o) for t in (parent, pr))
        sa, sb = sass(pa), sass(pb)
        ra, rb = resources(pa + ".log"), resources(pb + ".log")
        same = sum(1 for k in sb if k in sa and sa[k] == sb[k] and ra.get(k) == rb.get(k))
        only = sorted(set(sa) ^ set(sb))
        print(f"{o:14s} kernels {len(sb):4d}  identical {same:4d}  changed {len(sb) - same - len(set(sb) - set(sa)):4d}"
              f"  only in one build {len(only)}")
        for k in only:
            print(f"    only in {'parent' if k in sa else 'PR'}: {NAMES[k]}")
        for k in sorted(sb):
            if k in sa and (sa[k] != sb[k] or ra.get(k) != rb.get(k)):
                changed.append((o, k, changed_lines(sa[k], sb[k]), len(sb[k]), ra.get(k), rb.get(k)))
    print()
    print(f"changed kernels: {len(changed)}")
    print(f"{'object':10s} {'instr changed/total':>24s} {'regs':>9s} {'spill st/ld':>11s} {'CTAs/SM':>8s}  kernel")
    for o, k, n, tot, a, b in changed:
        name = NAMES[k]
        threads, cap = launch_shape(name)
        ca, cb = (min(ctas_by_regs(r[0], threads), cap) if r else 0 for r in (a, b))
        print(f"{o[:-2]:10s} {n:>11d} / {tot:<10d} {a[0]:>3d} -> {b[0]:<3d} {b[1]:>5d}/{b[2]:<5d} {ca:>3d} -> {cb:<3d} {name}")


if __name__ == "__main__":
    main(*sys.argv[1:3])
