"""Per-kernel SASS comparison of two builds of the library (cuobjdump -sass, no GPU needed).

    python tools/sass_diff.py OLD.so NEW.so [--map OLD_NAME_SUBSTR=NEW_NAME_SUBSTR ...] > profiles/<file>.txt

Each kernel's instruction stream is compared with addresses and encodings stripped.  A kernel whose template gained a
parameter gets a new mangled name; `--map` rewrites the old demangled name before matching, e.g. the pool kernels that
became templates on the row width: `--map "k_pool_head<__half>=k_pool_head<__half, 512>"`.  Prints one line per
kernel of OLD (identical / differs / missing) and the kernels only NEW has.  Exit status 1 if any OLD kernel differs or
is missing."""
from __future__ import annotations

import re
import subprocess
import sys


def kernels(lib: str) -> dict:
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m:
            body.append(re.sub(r"\s+", " ", m.group(1)))
    if name:
        funcs[name] = body
    names = list(funcs)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {d: funcs[n] for n, d in zip(names, dem)}


def main(argv):
    maps = []
    args = []
    i = 0
    while i < len(argv):
        if argv[i] == "--map":
            old, new = argv[i + 1].split("=", 1)
            maps.append((old, new))
            i += 2
        else:
            args.append(argv[i])
            i += 1
    old_lib, new_lib = args
    old, new = kernels(old_lib), kernels(new_lib)
    bad, matched = 0, set()
    for name in sorted(old):
        target = name
        for a, b in maps:
            target = target.replace(a, b)
        if target not in new:
            print(f"MISSING   {name}")
            bad += 1
            continue
        matched.add(target)
        same = old[name] == new[target]
        bad += not same
        print(f"{'identical' if same else 'DIFFERS  '} {len(old[name]):6d} instr  {name}" +
              (f"  ->  {target}" if target != name else ""))
    for name in sorted(set(new) - matched):
        print(f"new       {len(new[name]):6d} instr  {name}")
    print(f"# {len(old)} kernels in {old_lib.split('/')[-1]}: {len(old) - bad} identical, {bad} differ or are missing")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
