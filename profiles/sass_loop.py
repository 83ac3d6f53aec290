#!/usr/bin/env python
"""Code-size gauge of a kernel's main loop, from the built object or library alone (no GPU).

For each kernel named by a substring of its mangled name: the loop is the backward branch that
encloses the most instructions (for the replay kernels, the epoch loop).  Reported: the kernel's
and the loop's instruction count and bytes, the nested loops, the opcode census inside the loop,
every LDL / STL and CALL inside it, and the loop's instructions per source line (`nvdisasm -g`
line info; the line is the innermost inlined one).  The ~32 KB instruction cache of an SM is the
yardstick: a loop that does not fit stalls on instruction fetch (`no_instruction`) every trip.

    python profiles/sass_loop.py roskfpos_b200/csrc/kfpos_t6.o profiles/r03_t6_loop_after.txt \\
        t6_replay_kernelILb0ELb0ELi8ELb0ELi1ELb0E t6_replay_kernelILb0ELb0ELi16ELb0ELi1ELb0E
"""
import collections
import glob
import os
import re
import subprocess
import sys
import tempfile

FP64 = ("DFMA", "DMUL", "DADD", "DSETP", "DMNMX")
INS = re.compile(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
LINE = re.compile(r'\s*//## File "([^"]+)", line (\d+)')
LABEL = re.compile(r"^(\.L_x_\d+):")
TARGET = re.compile(r"`\((\.L_x_\d+)\)")


def functions(path):
    """{mangled name: [(address, text, 'file:line')]} of every function in the object / library."""
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(path)], cwd=tmp, check=True,
                       capture_output=True)
        for cubin in sorted(glob.glob(os.path.join(tmp, "*.cubin"))):
            txt = subprocess.run(["nvdisasm", "-g", "-c", cubin], capture_output=True, text=True, check=True).stdout
            name, src, labels = None, "?", {}
            for ln in txt.splitlines():
                if ln.startswith("\t.section\t.text."):
                    name = ln.split(".text.", 1)[1].split(",", 1)[0]
                    out[name] = []
                    continue
                if name is None:
                    continue
                m = LINE.match(ln)
                if m:
                    src = f"{os.path.basename(m.group(1))}:{m.group(2)}"
                    continue
                m = LABEL.match(ln)
                if m:
                    labels[m.group(1)] = len(out[name])
                    continue
                m = INS.match(ln)
                if m:
                    out[name].append([int(m.group(1), 16), m.group(2), src])
            # resolve branch targets to instruction indices (labels are per cubin)
            for fn in out.values():
                for ins in fn:
                    t = TARGET.search(ins[1])
                    if len(ins) == 3:
                        ins.append(labels.get(t.group(1)) if t else None)
    return out


def opcode(text):
    return re.sub(r"^@!?U?P[T\d]+\s+", "", text).split()[0].split(".")[0]


def report(name, ins, top):
    n = len(ins)
    back = [(i - t + 1, t, i) for i, (_, text, _, t) in enumerate(ins)
            if t is not None and t <= i and opcode(text) == "BRA"]
    back.sort(reverse=True)
    r = [f"## {name}", f"kernel: {n} instructions, {16 * n / 1024:.1f} KB"]
    if not back:
        return r + ["no backward branch", ""]
    size, lo, hi = back[0]
    loop = ins[lo:hi + 1]
    r.append(f"loop: {size} instructions = {16 * size / 1024:.1f} KB (backward branch {ins[hi][0]:#06x} -> {ins[lo][0]:#06x})")
    inner = [(s, a, b) for s, a, b in back[1:] if lo <= a and b <= hi and s >= 50]
    for s, a, b in inner[:6]:
        r.append(f"  nested loop: {s} instructions ({ins[b][0]:#06x} -> {ins[a][0]:#06x}, starts at {ins[a][2]})")
    ops = collections.Counter(opcode(t) for _, t, _, _ in loop)
    fp = sum(ops[k] for k in FP64)
    r.append(f"inside the loop: FP64 {fp}, MUFU {ops['MUFU']}, other {size - fp - ops['MUFU']}; "
             f"LDL {ops['LDL']}, STL {ops['STL']}, CALL {ops['CALL']}")
    r.append("opcode census of the loop:")
    r += [f"  {op:10s} {c:5d}  {100.0 * c / size:5.1f} %" for op, c in ops.most_common()]
    r.append("local memory and calls inside the loop:")
    r += [f"  {a:#06x}  {t:60s} {s}" for a, t, s, _ in loop if opcode(t) in ("LDL", "STL", "CALL")]
    lines = collections.Counter(s for _, _, s, _ in loop)
    r.append(f"loop instructions per source line (top {top} of {len(lines)}):")
    r += [f"  {c:5d}  {s}" for s, c in lines.most_common(top)]
    return r + [""]


def main():
    if len(sys.argv) < 4:
        sys.exit(__doc__)
    path, out, keys = sys.argv[1], sys.argv[2], sys.argv[3:]
    fns = functions(path)
    rows = [f"# {os.path.basename(path)}: epoch-loop gauge (profiles/sass_loop.py)", ""]
    for key in keys:
        hit = sorted(k for k in fns if key in k and not k.startswith("$"))
        if len(hit) != 1:
            sys.exit(f"{key}: {len(hit)} kernels match {hit[:8]}")
        rows += report(hit[0], fns[hit[0]], 40)
    with open(out, "w") as f:
        f.write("\n".join(rows))
    print("\n".join(r for r in rows if r.startswith(("#", "kernel", "loop:", "inside"))))


if __name__ == "__main__":
    main()
