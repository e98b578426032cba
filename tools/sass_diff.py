#!/usr/bin/env python3
"""Per-kernel SASS of two builds of libvnect_b200.so, compared instruction for instruction (no GPU needed):

    python tools/sass_diff.py OLD.so NEW.so

Uniform-register numbers are normalised (they differ between two builds of the same source).  A kernel template that
gained a defaulted trailing bool (postprocess_kernel's SCORES) is matched by its old name.  Lines that differ only in
which entry of constant bank 4 (the module's address table: vprintf and format strings) they refer to are counted
apart, since that table's order follows the set of instantiations in the module.  Exit status 1 if a pre-existing
kernel is missing or differs in any other way.
"""
import re
import subprocess
import sys


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
        elif cur is not None:
            m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
            if m:
                res[cur].append(re.sub(r"\bUR\d+\b", "UR", m.group(1)).strip())
    return res


def old_name(name):
    m = re.match(r"(_ZN5vnect18postprocess_kernelILin?\d+ELin?\d+ELb[01]E)Lb0E(EEvNS_10PostParamsE)", name)
    return m.group(1) + m.group(2) if m else name


def bank4(line):
    return re.sub(r"c\[0x4\]\[[^\]]*\]", "c4", line)


def main():
    old, new = functions(sys.argv[1]), {old_name(k): v for k, v in functions(sys.argv[2]).items()}
    bad, table_only = [], []
    for k, v in old.items():
        w = new.get(k)
        if w is None or len(w) != len(v):
            bad.append(k)
        elif w != v:
            diff = [(a, b) for a, b in zip(v, w) if a != b]
            ok = all(bank4(a) == bank4(b) or (a.startswith("MOV ") and re.sub(r"0x[0-9a-f]+", "I", a) ==
                                               re.sub(r"0x[0-9a-f]+", "I", b)) for a, b in diff)
            (table_only if ok else bad).append(k)
    print(f"{len(old)} pre-existing kernels: {len(old) - len(bad) - len(table_only)} identical, "
          f"{len(table_only)} differing only in constant-bank-4 table entries, {len(bad)} changed or missing")
    for k in bad:
        print("  CHANGED", k)
    print(f"{len(set(new) - set(old))} new kernels:")
    for k in sorted(set(new) - set(old)):
        print("  ", k)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
