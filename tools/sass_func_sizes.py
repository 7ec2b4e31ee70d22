"""Instructions and local-memory accesses (LDL / STL: spills, by-reference structs) of a kernel per SOURCE function, from
the line markers of `nvdisasm -g` — no GPU needed. With two libraries: only the functions that differ (A/B of a build).
usage: python tools/sass_func_sizes.py libA.so [libB.so] [--kernel sf_rollout_kernelILi0]"""
import os, re, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "spacefortress_b200", "csrc")
args = [a for a in sys.argv[1:] if not a.startswith("--")]
kernel = sys.argv[sys.argv.index("--kernel") + 1] if "--kernel" in sys.argv else "sf_rollout_kernelILi0"
args = [a for a in args if a != kernel]

def marks_of(fn):
    lines = open(os.path.join(SRC, fn)).read().split("\n")
    m = [(i + 1, re.search(r"(sf_\w+)\s*\(", l).group(1)) for i, l in enumerate(lines)
         if re.match(r"(template.*)?(__device__|__global__|SF_HD|static)", l) and re.search(r"(sf_\w+)\s*\(", l)]
    return m + [(len(lines) + 1, "end")]

MARKS = {fn: marks_of(fn) for fn in ("sf_render.cuh", "sf_step.cuh", "sf_kernels.cu", "sf_geom.h")}

def func(f, ln):
    if f not in MARKS:
        return f
    for (s0, nm), (s1, _) in zip(MARKS[f], MARKS[f][1:]):
        if s0 <= ln < s1:
            return nm
    return f + ":?"

def sizes(lib):
    d = tempfile.mkdtemp()
    subprocess.run("cd %s && cuobjdump -xelf all %s >/dev/null 2>&1 && for f in *.sm_100a.cubin; do nvdisasm -g -c $f; done > all.dis 2>/dev/null" % (d, os.path.abspath(lib)), shell=True)
    cur, cnt, spl, inside = None, {}, {}, False
    for ln in open(os.path.join(d, "all.dis")):
        m = re.match(r"^\s*\.text\.(\S+)", ln)
        if m:
            inside = kernel in m.group(1)
        if not inside:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
        if m:
            cur = (m.group(1).split("/")[-1], int(m.group(2)))
            continue
        if cur and re.search(r"^\s*/\*[0-9a-f]{4,}\*/\s+[A-Z@!]", ln):
            k = func(*cur)
            cnt[k] = cnt.get(k, 0) + 1
            if re.search(r"\b(LDL|STL)\b", ln):
                spl[k] = spl.get(k, 0) + 1
    return cnt, spl

a, sa = sizes(args[0])
b, sb = sizes(args[1]) if len(args) > 1 else (a, sa)
print("%-32s %8s %8s   %6s %6s   (kernel %s; total %d / %d instructions)" % ("function", "instr A", "instr B", "loc A", "loc B", kernel, sum(a.values()), sum(b.values())))
for k in sorted(set(a) | set(b), key=lambda k: -max(a.get(k, 0), b.get(k, 0))):
    if len(args) == 1 or a.get(k, 0) != b.get(k, 0) or sa.get(k, 0) != sb.get(k, 0):
        print("%-32s %8d %8d   %6d %6d" % (k, a.get(k, 0), b.get(k, 0), sa.get(k, 0), sb.get(k, 0)))
