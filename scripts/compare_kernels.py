"""Compare the kernels of two libfwgym.so builds: SASS kernel by kernel, and ptxas resources per entry function.

    python fixed-wing-gym_b200/build.py --force -v > a.log   # keep the .so beside its log, then the same for b
    python scripts/compare_kernels.py a.so a.log b.so b.log [--mask]

--mask compares the SASS with every constant-bank operand offset masked (c[0x0][...] kernel parameters, c[0x4][...]
the module's global-address slots; the encoding words are dropped, they hold the same offsets): a change that appends to a parameter struct moves the later parameters, and one
that adds a __device__ object moves the address slots, without changing a single instruction.

SASS bodies are compared with leading and trailing whitespace stripped: whichever function ends an ELF section picks up
two trailing blank lines, and which one that is depends on the instantiation order.  ptxas -v lines are grouped by the
entry function they follow, because helpers such as __internal_trig_reduction_slowpathd are reported once per kernel
under the same name.  Exit status 1 if a kernel present in both builds differs.
"""
import re
import subprocess
import sys


def sass(lib, mask=False):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"^\s*Function : (\S+)\s*$", out, flags=re.M)
    if mask:
        # (the encoding words in the trailing comments carry the same offsets)
        parts = [re.sub(r"/\* 0x[0-9a-f]{16} \*/", "", re.sub(r"c\[0x[04]\]\[0x[0-9a-f]+\]", "c[..][..]", p))
                 for p in parts]
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


def main(lib_a, log_a, lib_b, log_b, mask=False):
    bad = 0
    for what, a, b in (("SASS", sass(lib_a, mask), sass(lib_b, mask)), ("ptxas", resources(log_a), resources(log_b))):
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
    args = [a for a in sys.argv[1:] if a != "--mask"]
    if len(args) != 4:
        sys.exit(__doc__)
    sys.exit(main(*args, mask="--mask" in sys.argv[1:]))
