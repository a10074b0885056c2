#!/usr/bin/env python
"""Warp instructions of one pass of features_tc_kernel's dimension loop (one warp, one dimension, 64 window values) on the
path the bench workload takes for most dimensions: image rows staged in shared memory, two regions, no SHAF rule, not a
constant or dropped column, "%.4g" text emulation on.  Static count from the SASS of libhafgpu.so (runs without a GPU).

The path is walked from the head of the loop: at a conditional branch the walk takes the side whose code does not come
from a source line of the rare cases (third region, SHAF, constant / dropped column, image rows read from global memory,
padding dimensions), else it falls through; it stops where it branches back to the head.  Every block on the path is
printed with the source lines its instructions come from, so the walk can be checked by eye.

  python tools/ft_hot_loop_count.py [--lo] [-v]        (--lo: the three-product build, which also writes the lo tile)
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "haf_grasping_b200", "lib", "libhafgpu.so")
SRC = os.path.join(ROOT, "haf_grasping_b200", "csrc", "kernels.cuh")
# source text of the rare cases: a block with an instruction from one of these lines is off the counted path
COLD = ("const uint4 t2 = lds_v4(", "f.off[8] = (int)t2.x;", "for (int k = 8; k < 12; k++) c[k] = load_corner(",
        "rr[2] = __fmul_rn(f.w[2],", "const float sa = __fsub_rn(rr[1], rr[0])", "raw = (rr[1] > rr[0] && rr[1] > rr[2])",
        "const float c = (f.flags & 0x400)", "xf[t] = (nrows > 0 || valid[t]) ? c : 0.0f", "valid[t] ? fast_tier_value(gI[t]",
        "return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(I + idx0) + off_bytes);",
        "for (; dl < KP; dl += 8) put(dl, 0u, 0u);")
HEAD = "for (; dl < KD; dl += 8) {"


def source_lines():
    lines = open(SRC).read().splitlines()
    cold = {i + 1 for i, ln in enumerate(lines) if any(c in ln for c in COLD)}
    head = [i + 1 for i, ln in enumerate(lines) if HEAD in ln]
    if len(cold) < len(COLD) - 1 or len(head) != 1:
        raise SystemExit("kernels.cuh no longer has the source lines this count is keyed on")
    return cold, head[0]


def disassemble(lo):
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(["cuobjdump", "-xelf", "all", LIB], cwd=tmp, check=True, capture_output=True)
        cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
        sass = subprocess.run(["nvdisasm", "-g", os.path.join(tmp, cubin)], check=True, capture_output=True, text=True).stdout
    name = "_ZN4hafk18features_tc_kernelILb%dE" % (1 if lo else 0)
    insts, labels, line, inside = [], {}, 0, False
    for ln in sass.splitlines():
        if ln.startswith(".text."):
            inside = ln.startswith(".text." + name)
            continue
        if not inside:
            continue
        m = re.match(r'\s*//## File ".*kernels\.cuh", line (\d+)', ln)
        if m:
            line = int(m.group(1))
            continue
        if re.match(r'\s*//## File', ln):
            line = 0
            continue
        m = re.match(r"^(\.L_x_\d+):", ln)
        if m:
            labels[m.group(1)] = len(insts)
            continue
        m = re.match(r"\s*/\*([0-9a-f]+)\*/\s+(.*?)\s*;", ln)
        if m:
            insts.append((int(m.group(1), 16), m.group(2), line))
    if not insts:
        raise SystemExit("no SASS for " + name)
    return insts, labels


def walk(insts, labels, cold, head_line):
    def target(text):
        m = re.search(r"`\((\.L_x_\d+)\)", text)
        return labels[m.group(1)] if m else None

    def is_branch(text):
        return re.match(r"(@!?U?P\w+\s+)?BRA(\.U)?\s", text) is not None

    def block_end(i):   # index after the block starting at i (at the next branch or label)
        starts = set(labels.values())
        j = i
        while j < len(insts):
            if is_branch(insts[j][1]) or insts[j][1].startswith("EXIT"):
                return j + 1
            j += 1
            if j in starts:
                return j
        return j

    def has_cold(i):
        return any(insts[k][2] in cold for k in range(i, block_end(i)))

    # head: the target of the branch back to the loop's first block (the back edge is on the loop's own line)
    backs = [(i, target(t)) for i, (_, t, ln) in enumerate(insts) if ln == head_line and is_branch(t) and target(t) is not None and target(t) < i]
    if not backs:
        raise SystemExit("loop back edge not found")
    back_i, head = max(backs, key=lambda b: b[0] - b[1])
    path, i, seen = [], head, set()
    while True:
        if i in seen:
            raise SystemExit("walk revisited a block at %#x" % insts[i][0])
        seen.add(i)
        e = block_end(i)
        path.append((i, e))
        text = insts[e - 1][1]
        if e - 1 == back_i:
            break
        if is_branch(text):
            t = target(text)
            cond = text.startswith("@") or re.match(r"BRA\.U\s+!?UP\d", text) is not None
            if not cond:
                i = t
            elif has_cold(t):
                i = e
            elif has_cold(e):
                i = t
            else:
                i = e
        else:
            i = e
    return path


def main():
    lo, verbose = "--lo" in sys.argv, "-v" in sys.argv
    cold, head_line = source_lines()
    insts, labels = disassemble(lo)
    path = walk(insts, labels, cold, head_line)
    total, ops = 0, collections.Counter()
    for i, e in path:
        n = e - i
        total += n
        lines = sorted({insts[k][2] for k in range(i, e)})
        print("  block %#06x: %3d instructions, kernels.cuh lines %s" % (insts[i][0], n, ",".join(map(str, lines))))
        for k in range(i, e):
            ops[insts[k][1].split()[0] if not insts[k][1].startswith("@") else insts[k][1].split()[1]] += 1
            if verbose:
                print("      %#06x  %-5d %s" % (insts[k][0], insts[k][2], insts[k][1]))
    kind = "three-product" if lo else "one/two-product"
    print("features_tc_kernel (%s build): %d warp instructions per (warp, dimension) on the staged, two-region, text-emulation path"
          % (kind, total))
    print("  by opcode: " + ", ".join("%s %d" % kv for kv in ops.most_common()))


if __name__ == "__main__":
    sys.exit(main())
