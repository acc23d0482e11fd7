"""Compare the SASS of two builds of libshems_b200.so kernel by kernel: `cuobjdump -sass` of each, split per function, addresses
(the /*0000*/ column) dropped.  Prints the kernels only one build has, and every kernel both have
whose instructions differ.

    python tools/sass_diff.py OLD.so NEW.so
"""
import re
import subprocess
import sys


def functions(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    fns, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:   # anonymous-namespace names carry a hash of the source path: a build from another directory renames them
            name = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))
            fns[name] = []
        elif name and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            fns[name].append(re.sub(r"/\*[0-9a-f]{4}\*/", "", line.split(";")[0]).strip())
    return fns


def main(old, new):
    a, b = functions(old), functions(new)
    only_a, only_b = sorted(set(a) - set(b)), sorted(set(b) - set(a))
    changed = sorted(k for k in set(a) & set(b) if a[k] != b[k])
    print(f"kernels: {len(a)} old, {len(b)} new; same SASS: {len(set(a) & set(b)) - len(changed)}")
    print("only in old:", only_a or "none")
    print("only in new:", only_b or "none")
    print("changed:", changed or "none")
    return 1 if (only_a or changed) else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
