#!/usr/bin/env python
"""Compare the SASS of the kernels in two object files / shared libraries instruction by instruction, over whole functions.

    python tools/sass_equal.py OLD.o NEW.o [substring ...] ['OLD_NAME=NEW_NAME' ...]

Used when a change must leave GPU-validated kernels untouched (no GPU at hand).  Kernels are matched by demangled name without
the parameter list; trailing `false` template arguments are folded away on both sides, so `kernel<3, true, false, false>` in OLD is
matched with `kernel<3, true, false>` in NEW.  An argument `OLD_NAME=NEW_NAME` pairs a renamed instantiation explicitly, e.g.
'wb_table_scatter_kernel<2, true, true>=wb_table_scatter_kernel<2>'; NEW_NAME is then matched with nothing else.  Substring arguments restrict the comparison to kernels whose
OLD name contains one of them.  Exit code 1 if any compared kernel differs or is missing on either side."""
import re
import subprocess
import sys


def _key(demangled):
    name = re.sub(r"^void ", "", demangled.split("(", 1)[0])
    return re.sub(r"(, false)+>", ">", name)


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []; continue
        if cur and re.match(r"\s*/\*[0-9a-f]+\*/", line):           # instruction lines start with their offset, of any length
            funcs[cur].append(re.sub(r"\s+", " ", re.sub(r"/\*.*?\*/", "", line)).strip())
    names = list(funcs)
    demangled = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {_key(d): funcs[n] for n, d in zip(names, demangled)}


def main():
    args = sys.argv[3:]
    pairs = {_key(a.split("=", 1)[0]): _key(a.split("=", 1)[1]) for a in args if "=" in a}
    want = [a for a in args if "=" not in a]
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    bad, seen = 0, set()
    for k, v in sorted(old.items()):
        if want and not any(w in k for w in want):
            continue
        kn = pairs.get(k, k)
        if kn not in new or (k not in pairs and kn in pairs.values()):       # a NEW name claimed by a pair matches nothing else
            print(f"{k[:90]:90s} MISSING in {sys.argv[2]}"); bad += 1; continue
        seen.add(kn)
        same = v == new[kn]
        bad += 0 if same else 1
        shown = k if kn == k else f"{k} = {kn}"
        print(f"{shown[:90]:90s} {'identical' if same else 'DIFFERENT'} ({len(v)} / {len(new[kn])} instructions)")
    for kn in sorted(set(new) - seen):
        if want and not any(w in kn for w in want):
            continue
        print(f"{kn[:90]:90s} MISSING in {sys.argv[1]}"); bad += 1
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
