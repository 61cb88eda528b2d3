"""Compare two builds of the library kernel by kernel, without a GPU: registers (cuobjdump -res-usage), stack frame and spill
bytes (the -Xptxas -v log of each build: `python -m libzombsole_b200.build -v > log 2>&1`), SASS instruction count and
whether the SASS is identical (cuobjdump -sass, instruction text without the encoding words).

usage: python tools/compiler_report.py PARENT.so PARENT_PTXAS.log NEW.so NEW_PTXAS.log"""
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def res_usage(lib):
    lines = subprocess.run([CUOBJDUMP, "-res-usage", lib], capture_output=True, text=True, check=True).stdout.splitlines()
    out = {}
    for i, line in enumerate(lines):
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            out[m.group(1)] = int(re.search(r"REG:(\d+)", lines[i + 1]).group(1))
    return out


def sass(lib):
    out, cur = {}, None
    for line in subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/", line):
            out[cur].append(re.sub(r"\s*/\* 0x[0-9a-f]+ \*/", "", line).strip())
    return out


def spills(log):
    out, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out[cur] = tuple(int(v) for v in m.groups())
            cur = None
    return out


def main():
    p_lib, p_log, n_lib, n_log = sys.argv[1:5]
    builds = [(res_usage(lib), spills(log), sass(lib)) for lib, log in ((p_lib, p_log), (n_lib, n_log))]
    names = sorted(set(builds[0][0]) | set(builds[1][0]))
    pretty = dict(zip(names, subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()))
    short = {k: pretty[k].replace("void ", "").replace("(ZsParams, ZsIO)", "") for k in names}

    def cols(b, k):
        reg, sp, ss = b[0].get(k), b[1].get(k), b[2].get(k)
        if reg is None:
            return "-"
        st, ls, ll = sp if sp else (0, 0, 0)
        return "regs %3d stack %3d spill st %3d ld %3d | SASS %5d" % (reg, st, ls, ll, len(ss))

    old = [k for k in names if k in builds[0][0]]
    same = [k for k in old if k in builds[1][0] and all(b0[k] == b1.get(k) for b0, b1 in zip(builds[0], builds[1]) if k in b0)]
    print("kernels of the parent: %d; of them with identical registers, stack, spills and SASS in the new build: %d" % (len(old), len(same)))
    print("kernels only in the new build: %d" % len([k for k in names if k not in builds[0][0]]))
    print()
    for k in sorted(names, key=lambda k: short[k]):
        tag = "identical" if k in same else ("NEW" if k not in builds[0][0] else "DIFFERS")
        print("%-46s parent: %s" % (short[k], cols(builds[0], k)))
        print("%-46s this:   %s   %s" % ("", cols(builds[1], k), tag))


if __name__ == "__main__":
    main()
