#!/usr/bin/env python3
"""Static SASS statistics of the device functions inside a kernel image of a shared library (no GPU needed).
usage: python tools/sass_fn_stats.py lib.so kernel_substr function_substr [--dump]
       python tools/sass_fn_stats.py lib.so kernel_substr --table
--table lists every function of the kernel (the kernel body first, then its callees by address) with its SASS
instruction count and its LDL / STL (local memory: spills and stack), R2UR and LDS counts, and the kernel's totals."""
import collections, os, re, subprocess, sys, tempfile


def functions(lib, ksub):
    """[(start, size, name)] of the kernel body and of every callee symbol inside the kernel image matching ksub."""
    tmp = tempfile.mkdtemp()
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, capture_output=True)
    cubin = os.path.join(tmp, [f for f in os.listdir(tmp) if f.endswith(".cubin")][0])
    sym = subprocess.run(["readelf", "-sW", cubin], capture_output=True, text=True).stdout
    out = []
    for ln in sym.splitlines():
        p = ln.split()
        if len(p) >= 8 and p[3] == "FUNC" and ksub in p[7]:
            out.append((int(p[1], 16), int(p[2]), p[7]))
    return out


def kernel_sass(lib, ksub):
    """[(address, instruction text)] of the kernel image whose name contains ksub."""
    dis = subprocess.run(["cuobjdump", "-sass", os.path.abspath(lib)], capture_output=True, text=True).stdout
    inside = False; out = []
    for ln in dis.splitlines():
        if "Function :" in ln: inside = ksub in ln and "$" not in ln
        if not inside: continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", ln)
        if m: out.append((int(m.group(1), 16), m.group(2).strip()))
    return out


def opcode(txt):
    t = txt.split()
    return (t[1] if t[0].startswith("@") else t[0]).split(".")[0]


def short_name(sym):
    name = sym.split("$")[-1]
    dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip() or name
    dem = re.sub(r"\(.*\)$", "", dem).replace("xm::", "")
    return dem


def table(lib, ksub):
    fns = sorted(f for f in functions(lib, ksub) if "$" in f[2])
    sass = kernel_sass(lib, ksub)
    cols = ("LDL", "STL", "R2UR", "LDS")
    rows = []; inside = set()
    for start, size, sym in fns:
        ins = [(a, t) for a, t in sass if start <= a < start + size]
        if not ins: continue
        inside.update(a for a, t in ins)
        ops = collections.Counter(opcode(t) for a, t in ins)
        rows.append((short_name(sym), len(ins)) + tuple(ops[c] for c in cols))
    # the kernel's own body: every instruction outside the callees
    ops = collections.Counter(opcode(t) for a, t in sass if a not in inside)
    rows.insert(0, ("(kernel body)", sum(ops.values())) + tuple(ops[c] for c in cols))
    total = collections.Counter(opcode(t) for a, t in sass)
    w = max(len(r[0]) for r in rows)
    print("%-*s %7s %6s %6s %6s %6s" % (w, "function", "instr", *cols))
    for r in rows:
        print("%-*s %7d %6d %6d %6d %6d" % ((w,) + r))
    print("%-*s %7d %6d %6d %6d %6d" % (w, "whole kernel", len(sass), *(total[c] for c in cols)))


def one(lib, ksub, fsub, dump):
    rng = None
    for start, size, sym in functions(lib, ksub):
        if fsub in sym and "$" in sym: rng = (start, size); name = sym
    if rng is None: sys.exit("function not found")
    ops = collections.Counter(); n = 0; lines = []
    for a, txt in kernel_sass(lib, ksub):
        if rng[0] <= a < rng[0] + rng[1]:
            ops[opcode(txt)] += 1; n += 1; lines.append("%6x  %s" % (a, txt))
    print(name, "bytes", rng[1], "instructions", n)
    print(dict(ops.most_common(16)))
    if dump: print("\n".join(lines))


if __name__ == "__main__":
    if "--table" in sys.argv:
        table(sys.argv[1], sys.argv[2])
    else:
        one(sys.argv[1], sys.argv[2], sys.argv[3], "--dump" in sys.argv)
