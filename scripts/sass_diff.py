"""Compares the SASS of two builds of libhqgraft.so kernel by kernel, modulo instruction addresses and register numbers.

    python scripts/sass_diff.py OLD.so NEW.so

Runs `cuobjdump -sass` on both libraries (no GPU needed), splits the listings per function and normalises away the
`/*0123*/` address and `/* 0x... */` encoding comments and the register numbers (two builds of the same source differ in
the registers ptxas assigns in about half of the tcgen05 kernels).  Every function of OLD must have the identical
instruction sequence in NEW: under the same name, or - for a kernel that became a template instantiation - under a new name whose
body is identical.  Prints one line per function that changed or disappeared and a summary; exit status 1 if any did.
Functions that exist only in NEW (new instantiations) are counted, not compared.
"""
from __future__ import annotations

import re
import subprocess
import sys

_ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")
_ENC = re.compile(r"/\*\s*0x[0-9a-f]+\s*\*/")
_REG = re.compile(r"\b(UR|R|UP|P|B)(\d+)\b")


def erase_registers(body):
    """R12 -> R#, UR7 -> UR#, P3 -> P#, ...: two ptxas runs on the same source were seen to assign registers (uniform
    registers around the tcgen05.mma issue) differently; RZ / URZ / PT / UPT stay."""
    return tuple(_REG.sub(lambda m: m.group(1) + "#", ins) for ins in body)


def functions(lib: str) -> dict:
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name is not None:
                funcs[name] = tuple(body)
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        ins = _ENC.sub("", _ADDR.sub("", line)).strip()
        if ins and not ins.startswith(".") and not ins.startswith("-"):
            body.append(re.sub(r"\s+", " ", ins))
    if name is not None:
        funcs[name] = tuple(body)
    return {n: erase_registers(b) for n, b in funcs.items()}


def demangle(names):
    res = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return dict(zip(names, res.stdout.splitlines())) if res.returncode == 0 else {n: n for n in names}


def main(old_lib: str, new_lib: str) -> int:
    old, new = functions(old_lib), functions(new_lib)
    dm = demangle(sorted(set(old) | set(new)))
    new_only = {n: b for n, b in new.items() if n not in old}
    by_body = {}
    for n, b in new_only.items():
        by_body.setdefault(b, []).append(n)
    same = renamed = 0
    bad = []
    for n, b in sorted(old.items()):
        if n in new:
            if new[n] == b:
                same += 1
            else:
                bad.append(f"CHANGED  {dm[n]}  ({len(b)} -> {len(new[n])} instructions)")
        elif b in by_body:
            renamed += 1
            print(f"renamed, identical: {dm[n]}  ->  {dm[by_body[b][0]]}")
        else:
            bad.append(f"MISSING  {dm[n]}")
    for line in bad:
        print(line)
    print(f"{len(old)} functions in {old_lib}: {same} identical, {renamed} identical under a new name, {len(bad)} changed or "
          f"missing; {len(new_only) - renamed} new functions in {new_lib}")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        raise SystemExit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
