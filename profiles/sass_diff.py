#!/usr/bin/env python
"""Per-kernel comparison of two `cuobjdump -sass` dumps of the same object, with addresses and encodings stripped,
and the `-Xptxas -v` lines (registers, spills, shared memory) of each entry function.  A kernel of the new dump is
matched with the old one of the same name once a trailing template argument 0 and a trailing TanTables parameter are
dropped (the xyz instantiations of the kernels that gained a frame-kind parameter).
usage: sass_diff.py old.sass new.sass [new_ptxas.txt [old_ptxas.txt]]"""
import re
import subprocess
import sys


def demangle(name):
    return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()


def kernels(path):
    """{demangled name: [instruction text, ...]}"""
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = demangle(m.group(1))
            out[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*/\*", line)
        if cur and m:
            out[cur].append(m.group(1))
    return out


def old_name(name):
    return name.replace(", 0>", ">").replace(", nav::TanTables)", ")")


def ptxas_lines(path):
    """{demangled entry: 'N registers, S B smem, spills'}"""
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = demangle(m.group(1))
            continue
        if cur and "spill" in line:
            out[cur] = line.strip()
        elif cur and "Used" in line:
            out[cur] += "; " + line.split("Used", 1)[1].strip()
    return out


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    same = 0
    for name in sorted(old):
        got = [v for n, v in new.items() if n == name or old_name(n) == name]
        if not got:
            print(f"MISSING  {name}")
        elif got[0] == old[name]:
            same += 1
            print(f"same     {len(old[name]):5d} instructions  {name.split('(')[0]}")
        else:
            print(f"DIFFERS  {name.split('(')[0]}: {len(old[name])} -> {len(got[0])} instructions")
    print(f"{same} of {len(old)} kernels of the old dump compile to the same instructions")
    added = [n for n in new if n not in old and old_name(n) not in old]
    info = ptxas_lines(sys.argv[3]) if len(sys.argv) > 3 else {}
    print(f"{len(added)} new kernels:")
    for n in sorted(added):
        print(f"  {n.split('(')[0]}: {info.get(n, '')}")
    if len(sys.argv) > 4:  # the -Xptxas -v lines of every function of both builds, file-hash prefixes dropped
        strip = lambda d: {re.sub(r"_INTERNAL_[0-9a-f]+_", "_INTERNAL_", k): v for k, v in d.items()}
        old_info, new_info = strip(ptxas_lines(sys.argv[4])), strip(info)
        differ = sorted(k for k in old_info.keys() | new_info.keys() if old_info.get(k) != new_info.get(k))
        print(f"-Xptxas -v: {len(old_info) - len(differ)} of {len(old_info)} functions of the old build report the same"
              f" registers, stack, spills and shared memory; {len(new_info)} functions in the new build")
        for k in differ:
            print(f"  {k.split('(')[0]}: {old_info.get(k)} -> {new_info.get(k)}")


if __name__ == "__main__":
    main()
