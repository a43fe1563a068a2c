#!/usr/bin/env python3
"""Static instruction counts of the fused iteration's pass-1 step loops, no GPU needed.

Compiles stoch_gpmp_b200/csrc/sgpmp_iterate_split.cu for sm_100a with the library's flags (plus -Xptxas -v), disassembles
it with nvdisasm -gi and, for the Panda kernel <7,1,4,4> (the C4 shape) and the planar kernel <2,0,4,0>, prints:
  * ptxas registers and spill bytes of the kernel;
  * the SASS opcodes of one time step of the state warps' step loop (state_sweep) and, for Panda, of the link warps'
    step loop (link_sweep), as static counts over the loop body.  The loop is the one whose back-edge branch belongs to
    the `for (int t = t0; t < tend; ...)` statement of that role, in the instance the benchmark runs (for the state
    warps the plain sweep: in-kernel stream, no sample output).  Instructions that come from the eps-injection branch of
    `draw` or from `emit_row` are left out, should a counted loop contain them.
  * spill loads / stores (LDL / STL) inside each loop.

usage: python profiles/hot_loop_counts.py [--csrc DIR] [--keep DIR]
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVDISASM = os.path.join(os.path.dirname(NVCC), "nvdisasm")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xptxas", "-v"]
SRC = "sgpmp_iterate_split.cu"
# (kernel, mangled name, [(role, step loop, calls of the role's lambdas that the benchmark's path takes: (pattern, which match))])
#   Panda: no map, 5 obstacle spheres (examples/panda_environment.py);  planar: the byte occupancy map.  The state sweep is the
#   PLAIN instance (in-kernel stream, no sample output).
PLAIN = (r"state_sweep_mm\(std::true_type", 0)
KERNELS = [("<7,1,4,4>", "_ZN5sgpmp20iterate_split_kernelILi7ELi1ELi4ELi4EEEvNS_10CostParamsIfEENS_8IterArgsIfEE",
            [("state", 0, [(r"state_sweep\(std::integral_constant<int, -1>", 1), PLAIN]),
             ("link", 1, [(r"link_sweep\(std::integral_constant<int, 5>", 0)])]),
           ("<2,0,4,0>", "_ZN5sgpmp20iterate_split_kernelILi2ELi0ELi4ELi0EEEvNS_10CostParamsIfEENS_8IterArgsIfEE",
            [("state", 0, [(r"state_sweep\(std::integral_constant<int, 1>", 0), PLAIN])])]


def source_lines(path):
    """Line numbers of the two step-loop statements (state, link), the line ranges left out of the counts, and a function
    that finds the line of the n-th match of a pattern."""
    src = open(path).read().split("\n")
    loops = [i + 1 for i, l in enumerate(src) if re.search(r"for \(int t = t0; t < tend;", l)]
    if len(loops) != 2:
        raise SystemExit("expected two step loops (state, link) in %s, found lines %s" % (path, loops))

    def block(start_re, end_test):
        first = next(i for i, l in enumerate(src) if re.search(start_re, l))
        last = next(i for i in range(first + 1, len(src)) if end_test(src[i]))
        return (first + 1, last + 1)

    emit = block(r"auto emit_row = \[&\]", lambda l: l.strip() == "};")
    draw = next(i for i, l in enumerate(src) if re.search(r"auto draw = \[&\]", l))
    eps_first = next(i for i in range(draw, len(src)) if re.search(r"if \(eps\) \{", src[i]))
    eps_last = next(i for i in range(eps_first + 1, len(src)) if re.search(r"\} else \{", src[i]))

    def find(pattern, n):
        return [i + 1 for i, l in enumerate(src) if re.search(pattern, l)][n]

    return loops, [emit, (eps_first + 1, eps_last + 1)], find


def parse_function(listing, mangled):
    """[(opcode, chain)] and {label: index} of one function; chain = [(file, line), ...] innermost first."""
    head = ".text.%s:" % mangled
    start = listing.index(head)
    nxt = listing.find("\n.text.", start + len(head))
    body = listing[start: nxt if nxt >= 0 else len(listing)].split("\n")
    instrs, labels, chain, pending = [], {}, [], []
    for l in body:
        m = re.match(r'\s*//## File "([^"]*)", line (\d+)(?: inlined at "([^"]*)", line (\d+))?', l)
        if m:
            if not pending:
                pending.append((os.path.basename(m.group(1)), int(m.group(2))))
            if m.group(3):
                pending.append((os.path.basename(m.group(3)), int(m.group(4))))
            continue
        if pending:
            chain, pending = pending, []
        m = re.match(r"^(\.L_x_\d+):", l)
        if m:
            labels[m.group(1)] = len(instrs)
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(@!?U?P[T\d]+\s+)?([A-Z][A-Z0-9_.]*)(.*)", l)
        if m:
            tgt = re.search(r"`\((\.L_x_\d+)\)", m.group(3))
            instrs.append((m.group(2), chain, tgt.group(1) if tgt else None))
    return instrs, labels


def loop_body(instrs, labels, loop_line, via_lines):
    """Instruction index range of the innermost loop whose back-edge belongs to source line loop_line, inlined through every
    line of via_lines."""
    best = None
    for i, (op, chain, tgt) in enumerate(instrs):
        if op.startswith("BRA") and tgt in labels and labels[tgt] <= i and chain and chain[0] == (SRC, loop_line) \
                and all((SRC, v) in chain for v in via_lines):
            r = (labels[tgt], i)
            if best is None or r[1] - r[0] < best[1] - best[0]:
                best = r
    if best is None:
        raise SystemExit("no back-edge for %s:%d" % (SRC, loop_line))
    return best


def count(instrs, rng, excluded):
    ops = collections.Counter()
    for op, chain, _ in instrs[rng[0]: rng[1] + 1]:
        if any(f == SRC and any(a <= ln <= b for a, b in excluded) for f, ln in chain):
            continue
        ops[op] += 1
    return ops


def summary(ops):
    base = collections.Counter()
    for op, n in ops.items():
        base[op.split(".")[0]] += n
    wide = sum(n for op, n in ops.items() if op.startswith("IMAD.WIDE"))
    top = ", ".join("%s %d" % kv for kv in base.most_common(16))
    return sum(ops.values()), wide, ops.get("LDL", 0) + sum(n for op, n in ops.items() if op.startswith("LDL.")), \
        sum(n for op, n in ops.items() if op.split(".")[0] == "STL"), top


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--csrc", default=os.path.join(ROOT, "stoch_gpmp_b200", "csrc"), help="source directory to compile")
    ap.add_argument("--keep", default=None, help="directory for the cubin, the ptxas log and the SASS listing")
    a = ap.parse_args()
    out = a.keep or tempfile.mkdtemp(prefix="hot_loop_counts_")
    os.makedirs(out, exist_ok=True)
    src = os.path.join(a.csrc, SRC)
    cubin = os.path.join(out, "split.cubin")
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(a.csrc))), "include")
    r = subprocess.run([NVCC] + FLAGS + ["-I", inc, "-cubin", "-o", cubin, src], capture_output=True, text=True, cwd=a.csrc)
    if r.returncode:
        sys.exit(r.stdout + r.stderr)
    open(os.path.join(out, "ptxas.txt"), "w").write(r.stderr)
    listing = subprocess.run([NVDISASM, "-gi", "-c", cubin], capture_output=True, text=True, check=True).stdout
    open(os.path.join(out, "split.sass"), "w").write(listing)
    loops, excluded, find = source_lines(src)
    for name, mangled, roles in KERNELS:
        m = re.search(r"Function properties for %s\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                      r".*?Used (\d+) registers" % re.escape(mangled), r.stderr, re.S)
        print("iterate_split_kernel%s: %s registers, %s B spill stores, %s B spill loads" % (name, m.group(4), m.group(2), m.group(3)))
        instrs, labels = parse_function(listing, mangled)
        for role, loop, vias in roles:
            rng = loop_body(instrs, labels, loops[loop], [find(p, n) for p, n in vias])
            tot, wide, ldl, stl, top = summary(count(instrs, rng, excluded))
            print("  %-5s step loop: %3d instr/step, IMAD.WIDE %d, LDL %d, STL %d | %s" % (role, tot, wide, ldl, stl, top))


if __name__ == "__main__":
    main()
