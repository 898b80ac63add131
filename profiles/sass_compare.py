"""Compare the SASS of every kernel in two builds of libbeng.so, instruction by instruction.

    python profiles/sass_compare.py PARENT.so NEW.so

Kernels are compared by name.  builder_kernel gained a DELTA template argument after a parent that had none: a parent's
builder_kernel<T, R, C> is compared with the new build's <T, R, C, false>.  Kernels of the new build that have no
parent, such as the DELTA = true instantiations, are listed with their instruction count, registers, stack frame and
local memory beside those of their DELTA = false twin.  Constant-bank offsets are part of the compared text.  Needs
cuobjdump and c++filt, no GPU.
"""
import re
import subprocess
import sys


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return dict(zip(names, out))


def kernels(so):
    """-> {demangled name: [instruction text]}, {demangled name: {"REG": .., "STACK": .., "LOCAL": ..}}"""
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
    usage, name = {}, None
    out = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True, check=True).stdout
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL):(\d+)", line)}
    plain = demangle(list(res) + [k for k in usage if k not in res])
    return {plain[k]: v for k, v in res.items()}, {plain[k]: v for k, v in usage.items()}


def parent_name(name):
    """The name a kernel of the new build had in a parent without builder_kernel's DELTA argument."""
    m = re.match(r"(.*builder_kernel<\d+, \w+, \d+), false>(.*)", name)
    return m.group(1) + ">" + m.group(2) if m else name


def describe(sass, usage, name):
    u = usage.get(name, {})
    return f"{len(sass[name])} instructions, {u.get('REG')} registers, stack {u.get('STACK')} B, local {u.get('LOCAL')} B"


def main():
    (parent, _), (new, usage) = kernels(sys.argv[1]), kernels(sys.argv[2])
    delta_in_parent = not any(re.search(r"builder_kernel<\d+, \w+, \d+>", k) for k in parent)
    as_parent = {k if delta_in_parent else parent_name(k): k for k in new}  # parent's name -> this build's name
    same, added = 0, []
    for name in sorted(set(parent) | set(as_parent)):
        if name not in as_parent:
            print(f"only in parent: {name}")
        elif name not in parent:
            added.append(as_parent[name])
        elif parent[name] != new[as_parent[name]]:
            print(f"DIFFERENT: {name}: {len(parent[name])} -> {len(new[as_parent[name]])} instructions")
        else:
            same += 1
    print(f"{same} of {len(parent)} parent kernels have identical SASS")
    for name in added:
        print(f"new kernel: {name}: {describe(new, usage, name)}")
        twin = re.sub(r", true>(?=[^<>]*$)", ", false>", name)
        if twin != name and twin in new:
            print(f"    its DELTA = false twin: {describe(new, usage, twin)}")
    return 0 if same == len(parent) else 1


if __name__ == "__main__":
    sys.exit(main())
