#!/usr/bin/env python
"""Instruction counts of the march loop's paths in the inline-shading batch kernel, read from its SASS.

    python tools/sass_paths.py [build/obj/vr_kernels_16.o build/obj/vr_kernels_25.o ...]

For march_persistent_kernel<KBD, false, false, kOutLinear, 193> of every object given (default: the SH16 and SH25
objects of `make lib`) it runs `cuobjdump -sass` and prints, per path through one iteration of the march loop:

  empty   a sample whose first table fetch is a leaf with sigma <= threshold: the loop body with the extra-fetch
          loop and the shading block skipped, plus the loop tail up to the back edge
  fetch   one more round of the table descent (the inner loop of find_leaf_wide)
  shade   the shading block (the sigma test's taken side, up to where it rejoins the loop tail)

and the number of paired fp32 instructions (FFMA2 / FADD2 / FMUL2) in the march loop and in the whole kernel.

How the loop is found: the march loop is the smallest loop (backward branch) whose body holds a 256-bit colour-record
load; the extra-fetch loop is the backward branch inside it whose body holds a table load (LDG) and no record load;
the shading block is skipped by the first forward conditional branch after the extra-fetch loop whose target lies past
the first record load.  The empty path follows the straight line from the loop head and takes every forward branch
that skips the extra-fetch loop or the shading block.
"""
import json
import re
import subprocess
import sys

KERNEL = "_ZN3vrb23march_persistent_kernelILi{kbd}ELb0ELb0ELi0ELi193EEEvNS_9LaunchDevE"
INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
PAIRED = re.compile(r"\b(FFMA2|FADD2|FMUL2)\b")


def parse_sass(text):
    """[(address, instruction text without the trailing ';')] of a cuobjdump -sass listing"""
    insns = []
    for line in text.splitlines():
        m = INSN.match(line)
        if m:
            insns.append((int(m.group(1), 16), m.group(2)))
    return insns


def kernel_sass(obj, name):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", name, obj], check=True, capture_output=True, text=True).stdout
    insns = parse_sass(out)
    if not insns:
        raise SystemExit(f"{obj}: kernel {name} not found")
    return insns


def branch_target(text):
    m = re.search(r"\bBRA(?:\.\w+)*\s+(?:!?U?P\d+,\s*)?(0x[0-9a-f]+)", text)
    return int(m.group(1), 16) if m else None


def analyse(insns):
    addr = [a for a, _ in insns]
    pos = {a: i for i, a in enumerate(addr)}
    rec = [i for i, (_, t) in enumerate(insns) if re.search(r"\bLDG\S*\.256", t)]
    # loops: (head index, back-edge index)
    loops = []
    for i, (a, t) in enumerate(insns):
        tgt = branch_target(t)
        if tgt is not None and tgt <= a and tgt in pos:
            loops.append((pos[tgt], i))
    march = min((l for l in loops if any(l[0] <= r <= l[1] for r in rec)), key=lambda l: l[1] - l[0])
    h, e = march
    fetch = [l for l in loops if h < l[0] and l[1] < e and
             any(re.search(r"\bLDG\b", insns[k][1]) for k in range(l[0], l[1] + 1)) and
             not any(l[0] <= r <= l[1] for r in rec)]
    if len(fetch) != 1:
        raise SystemExit(f"expected one extra-fetch loop in the march loop, found {len(fetch)}")
    fh, fe = fetch[0]
    first_rec = min(r for r in rec if h <= r <= e)
    shade = None
    for i in range(fe + 1, first_rec):
        t = insns[i][1]
        tgt = branch_target(t)
        if tgt is not None and t.startswith("@") and tgt > addr[i] and pos.get(tgt, -1) > first_rec:
            shade = (i, pos[tgt])
            break
    if shade is None:
        raise SystemExit("shading branch not found")
    # empty path: straight line from the loop head, skipping the extra-fetch loop and the shading block
    n, i, seen = 0, h, set()
    while True:
        if i in seen:
            raise SystemExit("empty path does not reach the back edge")
        seen.add(i)
        n += 1
        if i == e:
            break
        t = insns[i][1]
        tgt = branch_target(t)
        if tgt is not None and tgt > addr[i] and tgt in pos:
            j = pos[tgt]
            skips = (i < fh and j > fe) or (i == shade[0])
            if skips or not t.startswith("@"):
                i = j
                continue
        i += 1
    loop_paired = sum(1 for k in range(h, e + 1) if PAIRED.search(insns[k][1]))
    return {
        "empty": n,
        "fetch": fe - fh + 1,
        "shade": shade[1] - shade[0] - 1,
        "paired_loop": loop_paired,
        "paired_kernel": sum(1 for _, t in insns if PAIRED.search(t)),
        "march_loop": [hex(addr[h]), hex(addr[e])],
    }


def main(argv):
    as_json = "--json" in argv
    objs = [a for a in argv if not a.startswith("--")] or ["build/obj/vr_kernels_16.o", "build/obj/vr_kernels_25.o"]
    res = {}
    for obj in objs:
        kbd = int(re.search(r"vr_kernels_(\d+)\.o$", obj).group(1))
        r = analyse(kernel_sass(obj, KERNEL.format(kbd=kbd)))
        res[f"SH{kbd}"] = dict(r, object=obj)
        if not as_json:
            print(f"SH{kbd:<3d} empty sample {r['empty']:4d}   extra fetch round {r['fetch']:3d}   shading block "
                  f"{r['shade']:4d}   paired fp32: {r['paired_loop']} in the march loop, {r['paired_kernel']} in "
                  f"the kernel   ({obj}, loop {r['march_loop'][0]}..{r['march_loop'][1]})")
    if as_json:
        print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main(sys.argv[1:])
