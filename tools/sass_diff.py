#!/usr/bin/env python3
"""Compares the SASS of the fp16 kernels of two builds of libfa_b200.so (or of two object files), function by function.

    python tools/sass_diff.py OLD.so NEW.so

Adding the element type as a template parameter (fp16 / bf16 instantiations of the same tcgen05 kernels) renames every
fp16 kernel, so names are demangled and normalised first: `<__half>` and a leading `__half, ` template argument are
dropped, and so is the return type that templates carry in their demangled names; the pair type `Pair<__half>` of the
vectorised passes reads as `__half2`. Every function of OLD must then have
a function of NEW with the same normalised name and byte-identical SASS. Functions only in NEW (the bf16
instantiations) are counted, not compared. Exit code 0 when nothing differs. Needs cuobjdump and c++filt; no GPU."""
import re
import subprocess
import sys


def functions(path):
    sass = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    out, name, body = {}, None, []
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = "\n".join(body)
            name, body = m.group(1), []
        elif name:
            if "Fatbin" in line:   # the next cubin of the library
                out[name] = "\n".join(body)
                name, body = None, []
            elif line.strip():
                body.append(line.rstrip())
    if name:
        out[name] = "\n".join(body)
    return out


def demangle(names):
    res = subprocess.run(["c++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout
    return res.splitlines()


def normalise(name):
    name = re.sub(r"^void ", "", name)
    name = re.sub(r"std::conditional<std::is_same<__half, __half>::value, __half2, __nv_bfloat162>::type", "__half2", name)
    name = name.replace("<__half>", "").replace("<__half, ", "<")
    return name


def main():
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    old_n = dict(zip(map(normalise, demangle(list(old))), old.values()))
    new_n = dict(zip(map(normalise, demangle(list(new))), new.values()))
    missing = [n for n in old_n if n not in new_n]
    differ = [n for n in old_n if n in new_n and old_n[n] != new_n[n]]
    only_new = [n for n in new_n if n not in old_n]
    print(f"{len(old_n)} functions in {sys.argv[1]}, {len(new_n)} in {sys.argv[2]}")
    print(f"identical: {len(old_n) - len(missing) - len(differ)}  differ: {len(differ)}  missing: {len(missing)}  "
          f"new only: {len(only_new)} ({sum('bfloat16' in n for n in only_new)} bf16)")
    for n in differ:
        print("DIFFERS:", n)
    for n in missing:
        print("MISSING:", n)
    for n in only_new:
        if "bfloat16" not in n:
            print("NEW (not bf16):", n)
    sys.exit(1 if missing or differ else 0)


if __name__ == "__main__":
    main()
