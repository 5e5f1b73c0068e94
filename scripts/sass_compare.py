"""Compares the device code of two builds of libgvcnn_sm100.so, kernel by kernel (cuobjdump -sass and -res-usage).

    python scripts/sass_compare.py OLD.so NEW.so

For a change that should leave every kernel as it was (a host-side refactor): each kernel present in both libraries
must have the same instruction text and the same registers, stack, shared and local memory.  A difference only in the
target offsets of BRA / CALL.REL is reported as such; any other difference fails.  Prints the kernels only in OLD
(dropped instantiations) and only in NEW, and exits non-zero when a common kernel differs or NEW has a kernel OLD lacks.
Names of kernels in anonymous namespaces carry a per-build hash, which is normalised away.
"""
import re
import subprocess
import sys

ANON = re.compile(r"\d*_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+")
INSN = re.compile(r"^\s+/\*([0-9a-f]{4,5})\*/\s+(.*?)\s*;?\s*/\*")


def norm(name):
    return ANON.sub(lambda m: "_GLOBAL__N__" + m.group(1), name)


def sass(so):
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = norm(m.group(1))
            funcs[cur] = []
            continue
        m = INSN.match(line)
        if cur and m:
            funcs[cur].append(m.group(2))
    return funcs


def res_usage(so):
    out = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            cur = norm(m.group(1))
        elif cur and "REG:" in line:
            res[cur] = " ".join(f for f in line.split() if f.split(":")[0] in ("REG", "STACK", "SHARED", "LOCAL"))
            cur = None
    return res


def branch_only(a, b):
    """True when the two instruction lists differ only in the target offsets of branches and relative calls."""
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if x == y:
            continue
        if not re.search(r"\b(BRA|CALL\.REL)", x):
            return False
        if re.sub(r"0x[0-9a-f]+\s*$", "", x) != re.sub(r"0x[0-9a-f]+\s*$", "", y):
            return False
    return True


def demangle(names):
    if not names:
        return []
    return subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True,
                          check=True).stdout.splitlines()


def main(old_so, new_so):
    old, new = sass(old_so), sass(new_so)
    rold, rnew = res_usage(old_so), res_usage(new_so)
    common = sorted(set(old) & set(new))
    only_old = sorted(set(old) - set(new))
    only_new = sorted(set(new) - set(old))
    failed, shifted = [], []
    for f in common:
        if rold.get(f) != rnew.get(f):
            failed.append((f, "resources %s -> %s" % (rold.get(f), rnew.get(f))))
        elif old[f] != new[f]:
            if branch_only(old[f], new[f]):
                shifted.append(f)
            else:
                failed.append((f, "instructions differ"))
    print("kernels: old %d, new %d, common %d" % (len(old), len(new), len(common)))
    print("identical instructions and resources: %d" % (len(common) - len(failed) - len(shifted)))
    print("branch / relative-call offsets only: %d" % len(shifted))
    for f in demangle(shifted):
        print("  ~ " + f)
    print("different: %d" % len(failed))
    for (f, why), d in zip(failed, demangle([f for f, _ in failed])):
        print("  ! %s: %s" % (d, why))
    print("only in old: %d" % len(only_old))
    for d in demangle(only_old):
        print("  - " + d)
    print("only in new: %d" % len(only_new))
    for d in demangle(only_new):
        print("  + " + d)
    return 1 if failed or only_new else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
