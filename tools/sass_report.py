"""SASS evidence for profiles/ (no GPU needed): per kernel the ptxas resource line, an opcode histogram, the global /
shared memory instruction variants (vector widths, cache hints), and the full listing (gzip when it is long).

    python tools/sass_report.py [--out profiles] [--prefix r02]
"""
import collections
import gzip
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "competitive-rl_b200", "libcrl_b200.so")
KERNELS = ["pong_step_kernel", "pong_raster_fast_kernelILi84ELb0", "pong_raster_fast_kernelILi84ELb1",
           "pong_raster_fast_kernelILi42ELb0", "pong_raster_fast_kernelILi42ELb1", "pong_raster_quad_kernelILi42",
           "car_step_kernel", "car_sensor_kernel", "car_collide_kernel", "car_render_kernel", "car_frame_setup_kernel", "car_frame_aux_kernel",
           "car_stack_shift_kernel", "car_reset_kernel", "car_pregen_kernel"]


def main():
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles")
    prefix = sys.argv[sys.argv.index("--prefix") + 1] if "--prefix" in sys.argv else "r02"
    sass = subprocess.run(["cuobjdump", "-sass", LIB], stdout=subprocess.PIPE, text=True).stdout
    res = subprocess.run(["cuobjdump", "-res-usage", LIB], stdout=subprocess.PIPE, text=True).stdout
    funcs = {}
    cur = None
    for ln in sass.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(ln)
    usage = {}
    lines = res.splitlines()
    for i, ln in enumerate(lines):
        m = re.search(r"Function (\S+):", ln)
        if m and i + 1 < len(lines):
            usage[m.group(1)] = lines[i + 1].strip()
    index = []
    for key in KERNELS:
        names = [n for n in funcs if key in n]
        if not names:
            continue
        name = names[0]
        body = funcs[name]
        ops = collections.Counter()
        mem = collections.Counter()
        for ln in body:
            m = re.search(r"/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", ln)
            if not m:
                continue
            op = m.group(1)
            ops[op.split(".")[0]] += 1
            if op.split(".")[0] in ("LDG", "STG", "LDS", "STS", "LDL", "STL", "ATOMG", "ATOMS", "RED", "LDC", "UBLKCP", "UTMASTG", "CCTL"):
                mem[op] += 1
        n_inst = sum(ops.values())
        short = key.replace("ILi", "_").replace("ELb0", "").replace("ELb1", "_ring")   # <DIM, RING> of the fast kernel
        fn = "%s_sass_%s.txt" % (prefix, short)
        head = ["# %s" % name, "# resources: %s" % usage.get(name, "?"), "# instructions: %d" % n_inst,
                "# opcode histogram: " + ", ".join("%s %d" % kv for kv in ops.most_common(28)),
                "# memory instructions: " + ", ".join("%s %d" % kv for kv in sorted(mem.items(), key=lambda kv: -kv[1])), ""]
        text = "\n".join(head + body) + "\n"
        if not ("raster_fast_kernelILi84" in key or "quad" in key):      # the two headline kernels stay plain text
            with gzip.open(os.path.join(out, fn + ".gz"), "wt") as f:
                f.write(text)
            with open(os.path.join(out, fn), "w") as f:
                f.write("\n".join(head) + "\n(full listing: %s.gz, %d lines)\n" % (fn, len(body)))
        else:
            with open(os.path.join(out, fn), "w") as f:
                f.write(text)
        index.append((short, n_inst, usage.get(name, "?"), dict(mem)))
        print(short, n_inst, usage.get(name, "?"))
    return index


if __name__ == "__main__":
    main()
