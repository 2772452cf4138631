"""Compare the SASS and resource usage of every kernel in two builds of the library.

  python tools/sass_compare.py BASE.so NEW.so [OLD=NEW ...]

Kernels are matched by demangled name without the anonymous-namespace prefix (which depends on the
source file name) and without the parameter list; OLD=NEW pairs match a renamed kernel.  For every
kernel of BASE it prints "same", "differs" (the instruction stream or REG / STACK / SHARED / LOCAL),
or "missing"; kernels only in NEW are listed as "new".  A differing kernel is marked "resources only"
when its instructions are identical, and "params only" when they match once the constant-bank
(kernel parameter) offsets are masked.  Under every other "differs" line it prints the resources
that changed and the per-opcode count changes (opcodes without their modifiers: DFMA, MUFU, ...).
Exit code 1 if any kernel of BASE differs or is missing.
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


def opcodes(body):
    return collections.Counter(re.sub(r"^@!?U?P\w+\s+", "", ins).split()[0].split(".")[0] for ins in body)


def delta(body, res, body2, res2):
    """What changed between two versions of a kernel: resources, then opcode counts."""
    out = [f"{k} {a} -> {b}" for k, a, b in zip(RES, res, res2) if a != b]
    c, c2 = opcodes(body), opcodes(body2)
    out += [f"{op} {c2[op] - c[op]:+d}" for op in sorted(set(c) | set(c2)) if c[op] != c2[op]]
    return ", ".join(out) or "same opcode counts and resources"


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
            if status == "differs" and len(new[twin]) == 1:
                print("          " + delta(body, res, *new[twin][0]))
    for name in sorted(set(new) - seen):
        print(f"new       {name}")
    print(f"{sum(len(v) for v in base.values())} base kernels, {bad} differ or are missing")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
