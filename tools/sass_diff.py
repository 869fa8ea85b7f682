"""dev tool: compare the SASS of every solve kernel in two builds of liba1mpc.so (cuobjdump -sass), kernel by kernel.

    python tools/sass_diff.py OLD.so NEW.so

Prints one line per kernel present in both builds (identical / DIFFERENT) and the kernels that only one build has.  The
warm-start kernels of the constant contact pattern gained a defaulted `bool EXT = false` template parameter when the
extended warm start was added, so their mangled names differ by `Lb0E`; they are matched under the new name."""
import re
import subprocess
import sys


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None and line.strip().startswith("/*"):   # instructions only (not the headers of the next ELF section)
            funcs[name].append(line.strip())
    return funcs


def canonical(name):
    # solve_kernel_warm<NS, N, WPC, LSM> -> solve_kernel_warm<NS, N, WPC, LSM, false>
    return re.sub(r"(17solve_kernel_warmILi\d+ELi\d+ELi\d+ELi\d+E)(EEv)", r"\1Lb0E\2", name)


def demangle(name):
    return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()


def main(old, new):
    a = {canonical(k): v for k, v in kernels(old).items()}
    b = kernels(new)
    rc = 0
    for k in sorted(set(a) | set(b)):
        if "solve_kernel" not in k:
            continue
        if k not in a:
            print("new only   ", demangle(k))
        elif k not in b:
            print("old only   ", demangle(k)); rc = 1
        elif a[k] == b[k]:
            print("identical  ", demangle(k), "(%d lines)" % len(a[k]))
        else:
            print("DIFFERENT  ", demangle(k)); rc = 1
    return rc


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
