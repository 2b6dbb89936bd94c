#!/usr/bin/env python3
"""Static SASS size of each phase of the physics tick (ex_tick in snake_exact_core.cuh) in the benchmarked kernel.

    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -DSNK_SCREEN -cubin -o /tmp/s.cubin \
        bullet_envs_b200/csrc/snake_exact.cu
    nvdisasm -gi /tmp/s.cubin > /tmp/s.sass
    python tools/sass_pass_sizes.py /tmp/s.sass

Every instruction is charged to the source line of ex_tick it comes from (for an inlined helper: the line of ex_tick that calls
it); the phases are told apart by the `// ---- ...` banners of ex_tick.  Static counts: no loop trip counts, no times."""
import re
import sys

CORE = "snake_exact_core.cuh"
# banner text of ex_tick -> phase that starts there (the phases run in this order)
BANNERS = [("pass 1: tip-ward", "pass 1"), ("free rigid motion about C", "rows + prologue"), ("projected Gauss-Seidel", "solver"),
           ("new base velocity", "base velocity"), ("pass 2: base-ward", "pass 2"), ("finish: Fz", "finish")]


def phase_lines(core_path):
    src = open(core_path).read().split("\n")
    start = next(i for i, s in enumerate(src) if "SNK_HD void ex_tick(" in s) + 1
    end = next(i for i in range(start, len(src)) if src[i].startswith("}")) + 1
    bounds = [(next(i for i in range(start, end) if b in src[i]) + 1, name) for b, name in BANNERS]
    return start, end, bounds


def sizes(sass_path, core_path, kernel="snk_hyb_step_kernelILb1ELb0ELb0E"):
    start, end, bounds = phase_lines(core_path)
    txt = open(sass_path).read()
    m = re.search(r"^\.text\.(_Z\w*%s\w*):$" % kernel, txt, re.M)
    body = txt[m.end():].split("\n//----")[0]
    out = {name: 0 for _, name in bounds}
    out["other"] = 0
    # nvdisasm -gi prints the inline chain of an instruction as consecutive `//##` lines, innermost first
    line, fresh = None, True
    for ln in body.split("\n"):
        m = re.search(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', ln)
        if m:
            if fresh:
                line, fresh = None, False
            for f, l in ((m.group(1), m.group(2)), (m.group(3), m.group(4))):
                if line is None and f and f.endswith(CORE) and start <= int(l) <= end:
                    line = int(l)
            continue
        fresh = True
        if not re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+\S", ln):
            continue
        ph = "other"
        if line is not None and start <= line <= end:
            for b, name in bounds:
                if line >= b:
                    ph = name
        out[ph] += 1
    return out


if __name__ == "__main__":
    import os
    core = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bullet_envs_b200", "csrc", CORE)
    for k, v in sizes(sys.argv[1], core).items():
        print("%-16s %6d" % (k, v))
