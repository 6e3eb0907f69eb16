"""Compare the kernels of two libfwgym.so builds: SASS kernel by kernel, and ptxas resources per entry function.

    python fixed-wing-gym_b200/build.py --force -v > a.log   # keep the .so beside its log, then the same for b
    python scripts/compare_kernels.py a.so a.log b.so b.log

SASS bodies are compared with leading and trailing whitespace stripped: whichever function ends an ELF section picks up
two trailing blank lines, and which one that is depends on the instantiation order.  ptxas -v lines are grouped by the
entry function they follow, because helpers such as __internal_trig_reduction_slowpathd are reported once per kernel
under the same name.  Exit status 1 if a kernel present in both builds differs.
"""
import re
import subprocess
import sys


def sass(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"^\s*Function : (\S+)\s*$", out, flags=re.M)
    return {name: body.strip() for name, body in zip(parts[1::2], parts[2::2])}


def resources(log):
    groups, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = groups.setdefault(m.group(1), [])
        elif cur is not None and ("ptxas info" in line or "bytes stack frame" in line) and "Compile time" not in line:
            cur.append(line.strip())
    return groups


def main(lib_a, log_a, lib_b, log_b):
    bad = 0
    for what, a, b in (("SASS", sass(lib_a), sass(lib_b)), ("ptxas", resources(log_a), resources(log_b))):
        print("%s: %d kernels vs %d" % (what, len(a), len(b)))
        for name in sorted(set(a) - set(b)):
            print("  only in the first:  %s" % name)
        for name in sorted(set(b) - set(a)):
            print("  only in the second: %s" % name)
        diff = [name for name in sorted(set(a) & set(b)) if a[name] != b[name]]
        for name in diff:
            print("  differs: %s" % name)
        print("  %d common, %d identical" % (len(set(a) & set(b)), len(set(a) & set(b)) - len(diff)))
        bad += len(diff)
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 5:
        sys.exit(__doc__)
    sys.exit(main(*sys.argv[1:]))
