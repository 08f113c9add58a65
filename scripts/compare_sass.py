"""Compare the machine code of two builds kernel by kernel.

    python scripts/compare_sass.py OLD NEW

OLD and NEW are builds of libpmdi_cuda.so, or cubins (the group module pmdi_spec_group.cubin, a run-time compiled
program written to a file).  For every kernel in either build it prints whether the SASS is the same and whether the
resource line (registers, stack, shared memory, ...) of `cuobjdump --dump-resource-usage` is the same, with the two
resource lines when they differ.  SASS is compared after stripping the instruction addresses, the encodings and the
mangled names of device functions (a renamed or merged device function gets a new name, not new code).  Exit status 1
when a kernel present in both builds differs.

A refactor of the sweep kernels that must not change what runs (and so not the per-step latency) keeps every
kernel "same" here.
"""
import os
import re
import shutil
import subprocess
import sys

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _run(*args):
    return subprocess.run([CUOBJDUMP, *args], capture_output=True, text=True, check=True).stdout


def sass(path):
    """kernel name -> normalised SASS lines"""
    out, name = {}, None
    for line in _run("-sass", path).splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        if name is None:
            continue
        line = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)       # address
        line = re.sub(r"/\* 0x[0-9a-f]{16} \*/", "", line)   # encoding
        line = re.sub(r"_Z\w+", "_Z", line)                  # mangled device-function names
        line = line.strip()
        if line:
            out[name].append(line)
    return out


def resources(path):
    """kernel name -> resource line"""
    out, name = {}, None
    for line in _run("--dump-resource-usage", path).splitlines():
        m = re.match(r"\s*Function (\S+):\s*$", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            out[name] = line.strip()
            name = None
    return out


def main(argv):
    if len(argv) != 3 or not all(os.path.exists(p) for p in argv[1:]):
        sys.exit(__doc__)
    old, new = argv[1], argv[2]
    s_old, s_new = sass(old), sass(new)
    r_old, r_new = resources(old), resources(new)
    names = sorted(set(s_old) | set(s_new))
    width = max(len(n) for n in names)
    print(f"{'kernel':<{width}}  {'sass':<9}  resources")
    bad = 0
    for n in names:
        if n not in s_old or n not in s_new:
            print(f"{n:<{width}}  {'only old' if n in s_old else 'only new':<9}  {r_old.get(n) or r_new.get(n)}")
            continue
        same_s = s_old[n] == s_new[n]
        same_r = r_old.get(n) == r_new.get(n)
        bad += not (same_s and same_r)
        res = "same  " + r_new.get(n, "") if same_r else f"DIFFERENT  old {r_old.get(n)}  new {r_new.get(n)}"
        if not same_s:
            diff = sum(a != b for a, b in zip(s_old[n], s_new[n])) + abs(len(s_old[n]) - len(s_new[n]))
            print(f"{n:<{width}}  {'DIFFERENT':<9}  {res}  ({diff} of {len(s_old[n])} lines)")
        else:
            print(f"{n:<{width}}  {'same':<9}  {res}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
