"""Compare the SASS of every kernel in two builds of libbeng.so, instruction by instruction.

    python profiles/sass_compare.py PARENT.so NEW.so

snake_kernel's DELTA template argument is dropped from the new build's names, so that each step kernel of the parent is
compared with its DELTA = false instantiation; the DELTA = true kernels are listed with their instruction counts.
Constant-bank offsets are part of the compared text.  Needs cuobjdump and c++filt, no GPU.
"""
import re
import subprocess
import sys


def kernels(so):
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            name = m.group(1)
            res[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(.*?);", line)
        if name and m:
            res[name].append(re.sub(r"\s+", " ", m.group(1)))
    names = list(res)
    plain = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return {p: res[k] for k, p in zip(names, plain)}


def main():
    parent, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    renamed = {}
    for name, sass in new.items():
        m = re.match(r"(.*snake_kernel<\d+, \w+, \w+), (true|false)>(.*)", name)
        if m and m.group(2) == "true":
            print(f"new kernel: {name}: {len(sass)} instructions")
            continue
        renamed[m.group(1) + ">" + m.group(3) if m else name] = sass
    same = 0
    for name in sorted(set(parent) | set(renamed)):
        if name not in parent or name not in renamed:
            print(f"only in {'parent' if name in parent else 'new'}: {name}")
        elif parent[name] != renamed[name]:
            print(f"DIFFERENT: {name}: {len(parent[name])} -> {len(renamed[name])} instructions")
        else:
            same += 1
    print(f"{same} of {len(parent)} parent kernels have identical SASS")
    return 0 if same == len(parent) == len(renamed) else 1


if __name__ == "__main__":
    sys.exit(main())
