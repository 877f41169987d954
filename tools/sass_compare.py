"""Instruction-for-instruction SASS comparison of the kernels two builds have in common.

Compiles nothing: give it two cubins (or objects / shared libraries) of the same source file, e.g. the parent commit's and the
working tree's, each built with ``nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -cubin``.  Kernels are
matched by demangled name; a template parameter added with a default (``bool kSelf = false``) makes the old instantiation's name
one ``, false`` longer, so a name is also matched with up to two trailing ``, false`` appended.  Instructions are compared with
addresses, symbol names and the anonymous-namespace hash removed.  Prints one line per old kernel (IDENTICAL / DIFFERENT /
MISSING) and then the kernels only the new build has.

    python tools/sass_compare.py OLD.cubin NEW.cubin [name-substring ...]
"""
import re
import subprocess
import sys


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?);?\s*/\*", line)
        if name and m:
            body.append(m.group(1))
    if name:
        funcs[name] = body
    names = list(funcs)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {clean(d): normalise(funcs[n]) for n, d in zip(names, dem)}


def clean(demangled):
    d = re.sub(r"_GLOBAL__N__[0-9a-f_]+", "", demangled)
    d = d.replace("ffr::(anonymous namespace)::", "").replace("ffr::", "")
    return re.sub(r"\(.*\)$", "", d).strip()


def normalise(instrs):
    # symbol names (relocations to functions / kernels carry the mangled, hash-bearing name)
    return [re.sub(r"\b_Z\w+", "SYM", re.sub(r"`\([^)]*\)", "SYM", i)) for i in instrs]


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    keys = sys.argv[3:]
    sel = lambda n: not keys or any(k in n for k in keys)
    matched = set()
    for name in sorted(n for n in old if sel(n)):
        cand = [name] + [name[:-1] + ", false" * k + ">" for k in (1, 2) if name.endswith(">")]
        hit = next((c for c in cand if c in new), None)
        if hit is None:
            print(f"{name} {len(old[name])} - MISSING")
            continue
        matched.add(hit)
        same = old[name] == new[hit]
        print(f"{name} {len(old[name])} {len(new[hit])} {'IDENTICAL' if same else 'DIFFERENT'}")
    for name in sorted(n for n in new if sel(n) and n not in matched):
        print(f"new: {name} {len(new[name])}")


if __name__ == "__main__":
    main()
