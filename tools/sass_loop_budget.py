#!/usr/bin/env python
"""Static instruction budget of the train step's two hot loops, on a CPU-only machine.

Compiles the train-path unit of one model (csrc/kge_train_inst.cu, -DKGE_TU_MODEL=<model>, default 3 = RotatE) for
sm_100a with -Xptxas -v, or reads an object built earlier, and for every row_kernel_split / entity_kernel instantiation
prints registers, stack and spills, and the opcode counts of its steady-state loop body:

  row_kernel_split   the candidate loop: the smallest backward-branch range holding the ring's mbarrier wait
                     (SYNCS.PHASECHK) and the distance math (MUFU.RSQ; for models without it, the largest such range)
  entity_kernel      the pair loop: found the same way

    python tools/sass_loop_budget.py [--model 3] [--obj FILE.o] [--filter 'row_kernel_split<3,0,8,2>'] [--all-ops]

A loop's count is static (instructions between the branch target and the backward branch), not a trace; the wait's
retry path, when ptxas moves it out of line, is not part of it.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "knowledgegraphembedding_b200", "csrc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-diag-suppress", "1886"]
KERNELS = ("row_kernel_split", "entity_kernel")
INSN = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(@!?U?P[0-9T]\s+)?([A-Z0-9_.]+)([^;]*);")
# opcode groups of the summary line (the rest is listed under 'other')
GROUPS = [("math", ("FADD", "FFMA", "FMUL", "MUFU", "FMNMX", "FSETP", "FSEL")),
          ("smem", ("LDS", "STS")),
          ("shfl", ("SHFL",)),
          ("copy/mbar", ("UBLKCP", "SYNCS", "ELECT", "R2UR", "UMOV", "UIADD3", "ULEA", "UISETP", "UPLOP3", "USEL",
                         "ULOP3", "USHF", "UIMAD", "ULDC", "LDCU", "VOTEU", "S2UR")),
          ("global", ("LDG", "STG", "REDG", "ATOMG", "RED")),
          ("branch", ("BRA", "BSSY", "BSYNC", "WARPSYNC", "EXIT", "CALL", "RET", "NOP"))]


def demangle(name):
    m = re.match(r"_ZN3kge(\d+)(\w+?)I(.*)EEv", name)
    if not m or len(m.group(2)) != int(m.group(1)):
        return name
    args = re.findall(r"L(i|b)(\d+)E", m.group(3))
    return "%s<%s>" % (m.group(2), ",".join(v for _, v in args))


def compile_unit(model, out_dir):
    obj = os.path.join(out_dir, "train_m%d.o" % model)
    res = subprocess.run([os.environ.get("NVCC", "nvcc")] + FLAGS + ["-Xptxas", "-v", "-DKGE_TU_MODEL=%d" % model, "-c",
                                                                     "kge_train_inst.cu", "-o", obj],
                         cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        sys.exit("nvcc failed:\n" + res.stdout + res.stderr)
    return obj, res.stderr


def ptxas_resources(log):
    """{mangled name: (registers, stack bytes, spill stores, spill loads)} from the -Xptxas -v log"""
    out, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line) or re.search(r"Function properties for (\w+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            r = out.get(cur, (0, 0, 0, 0))
            out[cur] = (r[0], int(m.group(1)), int(m.group(2)), int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            r = out.get(cur, (0, 0, 0, 0))
            out[cur] = (int(m.group(1)),) + r[1:]
    return out


def functions(obj):
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\w+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = INSN.match(line)
        if m and cur:
            funcs[cur].append((int(m.group(1), 16), m.group(3), m.group(4)))
    return funcs


def hot_loop(insns):
    """(start, end) of the loop body, see the module docstring"""
    addr = [a for a, _, _ in insns]
    loops = []
    for a, op, args in insns:
        if op.startswith("BRA") and not op.startswith("BRA.U.ANY"):
            t = re.search(r"0x([0-9a-f]+)\s*$", args.strip())
            if t and int(t.group(1), 16) <= a:
                loops.append((int(t.group(1), 16), a))
    def has(lo, hi, prefix):
        return any(lo <= x <= hi and op.startswith(prefix) for x, op, _ in insns)
    waits = [(lo, hi) for lo, hi in loops if has(lo, hi, "SYNCS.PHASECHK") and hi - lo > 0x400]
    rsq = [(lo, hi) for lo, hi in waits if has(lo, hi, "MUFU.RSQ")]
    if rsq:
        return min(rsq, key=lambda r: r[1] - r[0])
    return max(waits, key=lambda r: r[1] - r[0]) if waits else (addr[0], addr[-1])


def summarize(insns, lo, hi, all_ops):
    c = collections.Counter(op.split(".")[0] if not op.startswith(("MUFU", "SYNCS", "BRA")) else op
                            for a, op, _ in insns if lo <= a <= hi)
    total = sum(c.values())
    left = dict(c)
    parts = []
    for g, prefixes in GROUPS:
        n = 0
        for k in list(left):
            if k.startswith(prefixes):
                n += left.pop(k)
        parts.append("%s %d" % (g, n))
    parts.append("other %d" % sum(left.values()))
    lines = ["    loop 0x%x-0x%x: %d instructions (%s)" % (lo, hi, total, ", ".join(parts))]
    if all_ops:
        lines.append("    " + ", ".join("%s %d" % kv for kv in c.most_common()))
    else:
        key = ["MUFU.RSQ", "MUFU.EX2", "MUFU.RCP", "SHFL", "LDS", "FFMA2", "FADD2", "FMUL2", "REDG", "UBLKCP",
               "BRA.U.ANY", "ELECT", "R2UR", "S2R", "S2UR", "LDC", "LDCU", "STS", "STG", "LDL", "STL"]
        lines.append("    " + ", ".join("%s %d" % (k, c[k]) for k in key if c[k]))
    return lines


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--model", type=int, default=3, help="model id of include/kge_b200.h (3 = RotatE)")
    ap.add_argument("--obj", help="read this object instead of compiling (registers and spills are then not shown)")
    ap.add_argument("--filter", default="", help="only kernels whose demangled name contains this")
    ap.add_argument("--all-ops", action="store_true", help="list every opcode of the loop body")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        if args.obj:
            obj, res = args.obj, {}
        else:
            obj, log = compile_unit(args.model, tmp)
            res = ptxas_resources(log)
        funcs = functions(obj)
    for name in sorted(funcs, key=demangle):
        dn = demangle(name)
        if not dn.startswith(KERNELS) or args.filter not in dn:
            continue
        insns = funcs[name]
        r = res.get(name)
        rtxt = ("%d registers, %d B stack, %d B spill stores, %d B spill loads" % r) if r else "resources not known"
        print("%s: %d instructions, %s" % (dn, len(insns), rtxt))
        lo, hi = hot_loop(insns)
        print("\n".join(summarize(insns, lo, hi, args.all_ops)))


if __name__ == "__main__":
    main()
