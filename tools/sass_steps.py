#!/usr/bin/env python
"""Instruction count of the edge loops of SpMM kernels, read from the SASS of a cubin:
    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I include -cubin \\
         rgb-experiment_b200/csrc/spmm_inst_f32v.cu -o f32v.cubin
    python tools/sass_steps.py f32v.cubin 'spmm_rows_kernel<float, 4, 16, 1, 4, 0, 0>' ...
A loop is the range [target, branch] of a backward branch that holds a shared-memory load (the id broadcast) and at
least one global gather, with no other loop inside it.  Prints, per loop, the instructions, the gathers and the
predicated gathers.  A step that spans a whole batch (U >= G) is not a loop of its own and is not listed."""
import re
import subprocess
import sys

INS = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")


def kernels(cubin):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    cur, body = None, {}
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            body[cur] = []
            continue
        m = INS.search(line)
        if m and cur:
            body[cur].append((int(m.group(1), 16), m.group(2).strip()))
    return body


def loops(ins):
    found = []
    for addr, op in ins:
        m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)", op)
        if m and int(m.group(1), 16) < addr:
            lo = int(m.group(1), 16)
            body = [o for a, o in ins if lo <= a <= addr]
            if any("LDS" in o for o in body) and any("LDG" in o for o in body):
                found.append((lo, addr, body))
    return [(lo, hi, b) for lo, hi, b in found
            if not any(lo <= l2 and h2 <= hi and (l2, h2) != (lo, hi) for l2, h2, _ in found)]


def main():
    cubin, names = sys.argv[1], sys.argv[2:]
    body = kernels(cubin)
    demangled = {}
    for k in body:
        d = subprocess.run(["/usr/local/cuda/bin/cu++filt", k], capture_output=True, text=True).stdout.strip()
        demangled[k] = re.sub(r"\((?:int|bool)\)", "", d).replace("rgbmp::", "")
    for want in names:
        for k, d in demangled.items():
            if want not in d:
                continue
            print(d)
            for lo, hi, b in loops(body[k]):
                ld = [o for o in b if "LDG" in o]
                pred = [o for o in ld if o.startswith("@")]
                print(f"  loop 0x{lo:04x}-0x{hi:04x}: {len(b)} instructions, {len(ld)} gathers ({len(pred)} predicated)")


if __name__ == "__main__":
    main()
