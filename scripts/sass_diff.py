"""Compare the SASS of two builds of the library function by function.

    python scripts/sass_diff.py parent.so new.so

Runs `cuobjdump -sass` on both files and compares every function's instructions (encodings
included). The tag nvcc gives anonymous namespaces (_GLOBAL__N__<hash>_<file>_<hash>) depends on
the source text, so it is normalised first. Prints each function as identical or different, with
its instruction counts, and exits non-zero when any function differs or exists in one build only.
A refactor that claims to leave the kernels alone should show every function identical.
"""
import re
import subprocess
import sys

ANON_TAG = re.compile(r"_GLOBAL__N__[0-9a-f]{8}_\d+_\w+?_[0-9a-f]{8}")
INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/")


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in ANON_TAG.sub("_GLOBAL__N__", out).splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            if name in funcs:
                sys.exit(f"{path}: function {name} appears twice")
            funcs[name] = []
        elif name is not None and line.strip():
            funcs[name].append(line.rstrip())
    return funcs


def n_insn(lines):
    return sum(1 for l in lines if INSN.match(l))


def main():
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    a, b = functions(sys.argv[1]), functions(sys.argv[2])
    differ = 0
    for name in sorted(set(a) | set(b)):
        if name not in a or name not in b:
            where = sys.argv[2] if name in b else sys.argv[1]
            print(f"ONLY IN {where}  {name}")
            differ += 1
        elif a[name] == b[name]:
            print(f"identical  {n_insn(a[name]):7d}          {name}")
        else:
            print(f"DIFFERENT  {n_insn(a[name]):7d} -> {n_insn(b[name]):<7d} {name}")
            differ += 1
    print(f"{len(set(a) | set(b))} functions, {differ} different")
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
