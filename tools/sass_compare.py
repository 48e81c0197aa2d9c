#!/usr/bin/env python
"""tools/sass_compare.py OLD.so NEW.so -- compare the machine code (cuobjdump -sass) of every kernel of two
libcavb200.so builds, e.g. the parent commit's and this one's.

Instructions are compared without addresses and encodings.  Kernels are matched by demangled name; a kernel whose
parameter list changed is matched by its name without the parameter list when that is unique (k_track_record gained
parameters and a flags word); a harness kernel that gained a trailing bool template parameter (nve.cu: MASK, BATH) and a
trailing parameter of a new type is matched to its parent by dropping both when the new parameter is false.  Prints
SAME / DIFF / NEW / GONE lines and a count."""
import re
import subprocess
import sys

# the kernels whose template list grew by one bool in this change, and the parameter type that came with it
GROWN = r"k_nvt_one|k_nvt_two|k_md_one|k_md_fused"
NEW_PARAM = ", cavb::BathIn)"


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    fns, cur, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if cur:
                fns[cur] = body
            cur, body = m.group(1), []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s*(.*?);", line)
        if cur is not None and m:
            body.append(m.group(1).strip())
    if cur:
        fns[cur] = body
    names = list(fns)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {d: fns[n] for n, d in zip(names, dem)}


def parent_name(n):
    m = re.match(r"(.*cavb::(?:%s)<.*), (true|false)>(\(.*)" % GROWN, n)
    if not m:
        return n
    return (m.group(1) + ">" + m.group(3).replace(NEW_PARAM, ")")) if m.group(2) == "false" else None


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    same = diff = 0
    matched = set()
    by_stem = {}
    for p in old:
        by_stem.setdefault(p.split("(")[0], []).append(p)
    for n, body in sorted(new.items()):
        p = n
        if p not in old:
            stem = by_stem.get(n.split("(")[0], [])
            p = stem[0] if len(stem) == 1 and stem[0] not in new else parent_name(n)
        if p is None:
            print(f"NEW   {n.split('(')[0]}  ({len(body)} instructions)")
            continue
        if p not in old:
            print(f"NEW?  {n.split('(')[0]}  (no parent of that name)")
            diff += 1
            continue
        matched.add(p)
        if old[p] == body:
            same += 1
            if p != n:
                print(f"SAME  {p.split('(')[0]} -> {n.split('(')[0]} {len(body)}")
        else:
            diff += 1
            print(f"DIFF  {n.split('(')[0]}  parent {len(old[p])} vs {len(body)} instructions")
    for p in old:
        if p not in matched:
            print(f"GONE  {p.split('(')[0]}")
            diff += 1
    print(f"{same} kernels identical to the parent, {diff} different, {len(old)} kernels in the parent, {len(new)} now")
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main())
