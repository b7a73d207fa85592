#!/usr/bin/env python
"""Compare the SASS of two builds of the library kernel by kernel (cuobjdump, no GPU needed).

    python tools/sass_diff.py OLD.so NEW.so [--map OLD=NEW ...]

Kernels pair by demangled name without return type and parameter list (`vadb::fused_kernel<2, 2>`); --map pairs a
renamed kernel, e.g. --map 'vadb::tree_rows_kernel=vadb::rows_kernel<vadb::TreeArg>'.  For each pair the tool prints
whether the instruction text and the REG / SHARED / STACK / LOCAL of -res-usage are identical, and the first
instruction that differs.  Exit status 1 on any difference or on a kernel without a partner."""
import argparse
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
RES_KEYS = ("REG", "SHARED", "STACK", "LOCAL")


def _run(args):
    exe = CUOBJDUMP if os.path.isfile(CUOBJDUMP) else "cuobjdump"
    return subprocess.run([exe] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True).stdout


def _demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), stdout=subprocess.PIPE, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def _key(demangled):
    """`void vadb::k<1, 2>(vadb::P, int)` -> `vadb::k<1, 2>`: the parameter list's spelling may change with a rename."""
    s = demangled[5:] if demangled.startswith("void ") else demangled
    depth = 0
    for i, c in enumerate(s):
        if c == "<":
            depth += 1
        elif c == ">":
            depth -= 1
        elif c == "(" and depth == 0:
            return s[:i]
    return s


def load(lib):
    """{key: (instructions, resources)} of every kernel in lib."""
    code, fn = {}, None
    for line in _run(["-sass", lib]).splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            fn = m.group(1)
            code[fn] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m and fn:
            code[fn].append(" ".join(m.group(1).split()))
    res = {}
    for fn, vals in re.findall(r"Function (\S+):\s*\n\s*(.*)", _run(["-res-usage", lib])):
        kv = dict(re.findall(r"(\w+(?:\[\d+\])?):(\d+)", vals))
        res[fn] = {k: int(kv.get(k, 0)) for k in RES_KEYS}
    names = _demangle(sorted(code))
    out = {}
    for fn, insns in code.items():
        k = _key(names[fn])
        if k in out:
            raise SystemExit("%s: two kernels named %s" % (lib, k))
        out[k] = (insns, res.get(fn, {}))
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--map", action="append", default=[], metavar="OLD=NEW",
                    help="pair kernel OLD of the old build with kernel NEW of the new build")
    a = ap.parse_args(argv)
    ren = dict(m.split("=", 1) for m in a.map)
    old, new = load(a.old), load(a.new)
    bad = 0
    used = set()
    for k in sorted(old):
        nk = ren.get(k, k)
        label = k if nk == k else "%s -> %s" % (k, nk)
        if nk not in new:
            print("MISSING   %s" % label)
            bad += 1
            continue
        used.add(nk)
        (oi, orr), (ni, nr) = old[k], new[nk]
        if oi == ni and orr == nr:
            print("identical %s (%d instructions)" % (label, len(oi)))
            continue
        bad += 1
        print("DIFFERENT %s" % label)
        if orr != nr:
            print("    resources: %s -> %s" % (orr, nr))
        if oi != ni:
            i = next((j for j, (x, y) in enumerate(zip(oi, ni)) if x != y), min(len(oi), len(ni)))
            print("    %d vs %d instructions; first difference at #%d:" % (len(oi), len(ni), i))
            print("      - %s" % (oi[i] if i < len(oi) else "(end)"))
            print("      + %s" % (ni[i] if i < len(ni) else "(end)"))
    for k in sorted(set(new) - used):
        print("NEW       %s" % k)
        bad += 1
    print("%d old kernels, %d new kernels, %d problem(s)" % (len(old), len(new), bad))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
