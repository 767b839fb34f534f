"""Compare the SASS of two builds of libraymond_cuda.so, kernel by kernel.

    python scripts/sass_diff.py OLD.so NEW.so

Splits `cuobjdump -sass` of each library into one listing per kernel and compares the instruction text of every kernel of
OLD with the kernel of NEW that stands for the same instantiation: the kernel of the same name, or, for an OLD built before
k_shade gained its trailing template flag ENV and DevEnv parameter (the environment map), k_shade<F, P, K, L> of OLD is
k_shade<F, P, K, L, false> of NEW.  Likewise for an OLD built before the colour textures gave k_shade the flag TEX and a DevTex
parameter: k_shade<F, P, K, L, E> of OLD is k_shade<F, P, K, L, E, false> of NEW, and k_aov of OLD is k_aov<false>.
Prints one line per kernel of OLD and the kernels only NEW has; exits 1 when any kernel of OLD differs or is missing.
"""
from __future__ import annotations

import re
import shutil
import subprocess
import sys


def cuobjdump() -> str:
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand:
            return cand
    raise RuntimeError("cuobjdump not found")


def kernels(lib: str) -> dict:
    text = subprocess.run([cuobjdump(), "-sass", lib], check=True, capture_output=True, text=True).stdout
    out, name, body = {}, None, []
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = "\n".join(body)
            # kernels in an anonymous namespace carry a hash of the build path: drop it
            name, body = re.sub(r"_GLOBAL__N__[0-9a-f]{8}_(\d+_\w+?_cu)_[0-9a-f]{8}", r"_GLOBAL__N__\1", m.group(1)), []
        elif name and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            body.append(line.strip())
    if name:
        out[name] = "\n".join(body)
    return out


def old_name(new: str):
    """The OLD kernel a NEW one stands for (None: new instantiation)."""
    m = re.match(r"(_ZN2rm7k_shadeILb[01]ELi[01]ELb[01]ELb[01]ELb[01])ELb([01])(EEEv.*jjNS_6DevEnvE)NS_6DevTexE$", new)
    if m:
        return m.group(1) + m.group(3) if m.group(2) == "0" else None
    m = re.match(r"_ZN2rm5k_aovILb([01])EEEv(.*Pd)NS_6DevTexE$", new)
    if m:
        return "_ZN2rm5k_aovE" + m.group(2) if m.group(1) == "0" else None
    m = re.match(r"(_ZN2rm7k_shadeILb[01]ELi[01]ELb[01]ELb[01])ELb([01])(EEEv.*jj)NS_6DevEnvE$", new)
    if m:
        return m.group(1) + m.group(3) if m.group(2) == "0" else None
    return new


def main(old_lib: str, new_lib: str) -> int:
    old, new = kernels(old_lib), kernels(new_lib)
    by_old = {n: n for n in new if n in old}
    for n in new:
        o = old_name(n)
        if o is not None and o in old and o not in by_old:
            by_old[o] = n
    bad = 0
    for o in sorted(old):
        n = by_old.get(o)
        if n is None:
            print(f"MISSING    {o}")
            bad += 1
        elif old[o] != new[n]:
            print(f"DIFFERENT  {o}  ->  {n}")
            bad += 1
        else:
            lines = old[o].count("\n") + 1
            print(f"identical  {o}" + (f"  ->  {n}" if n != o else "") + f"  ({lines} SASS lines)")
    for n in sorted(set(new) - set(by_old.values())):
        print(f"new        {n}")
    print(f"{len(old)} kernels of the old build, {bad} differ or are missing")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
