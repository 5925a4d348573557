"""Compare the kernels of two builds of the same library, function by function.

    python profiles/compare_sass.py [--rename OLDNAME=NEWNAME ...] OLD.so NEW.so [OLD2.so NEW2.so ...]

For each pair, `cuobjdump -sass` and `cuobjdump -res-usage` are run on both libraries and every
function is compared by its mangled name: the SASS instructions (with their encodings) and the
resource line (registers, stack, shared and local memory).  Printed per pair: the number of
identical functions, the functions whose SASS or resources differ, and the functions that exist
in only one of the two builds.  --rename compares a kernel that was renamed under its new name: every
occurrence of OLDNAME in a function name of the old build is replaced by NEWNAME (mangled names,
e.g. 20rp_user_point_kernel=15rp_point_kernel).  Exit status 1 if any function differs or is missing.
"""
import re
import subprocess
import sys


def _sass(lib):
    """{function: [instruction lines]} of the sm_100a code in `lib`."""
    out = subprocess.run(["cuobjdump", "-sass", "-arch", "sm_100a", lib], capture_output=True, text=True,
                         check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            if cur in funcs:  # the same kernel in two translation units: compare both copies
                cur = cur + "#%d" % sum(k.split("#")[0] == m.group(1) for k in funcs)
            funcs[cur] = []
        elif cur and line.strip().startswith("/*"):
            funcs[cur].append(line.strip())
    return funcs


def _res(lib):
    """{function: resource-usage line} of the sm_100a code in `lib`."""
    out = subprocess.run(["cuobjdump", "-res-usage", "-arch", "sm_100a", lib], capture_output=True, text=True,
                         check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            cur = m.group(1)
            if cur in res:
                cur = cur + "#%d" % sum(k.split("#")[0] == m.group(1) for k in res)
        elif cur and "REG:" in line:
            res[cur] = line.strip()
            cur = None
    return res


def _renamed(d, renames):
    for a, b in renames:
        d = {k.replace(a, b): v for k, v in d.items()}
    return d


def compare(old, new, renames=()):
    so, sn = _renamed(_sass(old), renames), _sass(new)
    ro, rn = _renamed(_res(old), renames), _res(new)
    same = [f for f in so if f in sn and so[f] == sn[f] and ro.get(f) == rn.get(f)]
    differ = [f for f in so if f in sn and f not in same]
    gone = sorted(set(so) - set(sn))
    added = sorted(set(sn) - set(so))
    print("%s -> %s: %d functions identical" % (old, new, len(same)))
    for f in differ:
        print("  differs: %s (%d -> %d instructions; %s -> %s)" % (f, len(so[f]), len(sn[f]), ro.get(f), rn.get(f)))
    for f in gone:
        print("  only in old: " + f)
    for f in added:
        print("  only in new: " + f)
    return not (differ or gone or added)


if __name__ == "__main__":
    args, renames = sys.argv[1:], []
    while args[:1] == ["--rename"] and len(args) > 1:
        renames.append(tuple(args[1].split("=", 1)))
        args = args[2:]
    if not args or len(args) % 2:
        sys.exit(__doc__)
    ok = [compare(args[i], args[i + 1], renames) for i in range(0, len(args), 2)]
    sys.exit(0 if all(ok) else 1)
