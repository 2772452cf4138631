"""Compare the SASS and resource usage of every kernel in two builds of the library.

  python tools/sass_compare.py BASE.so NEW.so [OLD=NEW ...]

Kernels are matched by demangled name without the anonymous-namespace prefix (which depends on the
source file name) and without the parameter list; OLD=NEW pairs match a renamed kernel.  For every
kernel of BASE it prints "same", "differs" (the instruction stream or REG / STACK / SHARED / LOCAL),
or "missing"; kernels only in NEW are listed as "new".  A differing kernel is marked "resources only"
when its instructions are identical, and "params only" when they match once the constant-bank
(kernel parameter) offsets are masked.  Exit code 1 if any kernel of BASE differs or is missing.
"""
import collections
import re
import subprocess
import sys

RES = ("REG", "STACK", "SHARED", "LOCAL")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return {n: re.sub(r"^void |\(anonymous namespace\)::", "", d).split("(")[0] for n, d in zip(names, out)}


def kernels(so):
    """name -> list of (instructions, resources); a name can occur once per translation unit."""
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    code, cur = collections.defaultdict(list), None
    for ln in sass.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = []
            code[m.group(1)].append(cur)
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", ln)
        if m and cur is not None:
            cur.append(m.group(1))
    res = collections.defaultdict(list)
    usage = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True, check=True).stdout
    for name, line in re.findall(r"Function (\S+):\n\s*(.*)", usage):
        res[name].append(tuple(re.search(rf"\b{k}:(\d+)", line).group(1) for k in RES))
    names = demangle(list(code))
    out = collections.defaultdict(list)
    for mangled, bodies in code.items():
        out[names[mangled]] += zip(bodies, res[mangled])
    return out


def masked(body):
    return [re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", ins) for ins in body]


def main():
    base, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    renamed = dict(a.split("=", 1) for a in sys.argv[3:])
    bad, seen = 0, set()
    for name in sorted(base):
        twin = renamed.get(name, name)
        seen.add(twin)
        if twin not in new:
            print(f"missing   {name}")
            bad += 1
            continue
        for body, res in base[name]:
            if any(body == b and res == r for b, r in new[twin]):
                status = "same"
            else:
                bad += 1
                if any(body == b for b, _ in new[twin]):
                    status = "differs (resources only)"
                elif any(masked(body) == masked(b) for b, _ in new[twin]):
                    status = "differs (params only)"
                else:
                    status = "differs"
            print(f"{status:9s} {name}" + (f" -> {twin}" if twin != name else "") + f"  ({len(body)} instructions)")
    for name in sorted(set(new) - seen):
        print(f"new       {name}")
    print(f"{sum(len(v) for v in base.values())} base kernels, {bad} differ or are missing")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
