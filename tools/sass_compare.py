"""Compare the machine code of two builds of libaerobulk_gpu.so function by function.

    python tools/sass_compare.py [--ignore-offsets] OLD.so NEW.so      (or two saved `cuobjdump -sass` listings)

Splits `cuobjdump -sass` per function, drops the address comments and the fatbin headers (which name the source path),
and compares by function name.  Prints the number of identical functions and instructions, then every function that
differs, is gone or is new.  Exit status 1 when a function of OLD differs or is gone.

--ignore-offsets also drops the offsets into constant bank 3 (the __constant__ tables: c[0x3][0x1f0], c[0x3][RZ] and
c[0x3][R26+0x8] read as c[0x3][_], c[0x3][_] and c[0x3][R26+_]), the instruction encodings and the spacing, so that two
builds whose only difference is where the tables sit in the bank compare identical.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import sys

_HEADER = re.compile(r"^(Fatbin|code for|arch =|code version|host =|compile_size|identifier =|\.section|\.headerflags)")
_BANK3 = re.compile(r"c\[0x3\]\[(?:RZ|(U?R\d+))?(?:\+?-?0x[0-9a-f]+)?\]")
_ENCODING = re.compile(r"/\* 0x[0-9a-f]{16} \*/")


def _bank3(m: re.Match) -> str:
    return f"c[0x3][{m.group(1)}+_]" if m.group(1) else "c[0x3][_]"


def _listing(path: str) -> str:
    if not path.endswith(".so"):
        return open(path).read()
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    return subprocess.run([exe, "-sass", path], capture_output=True, text=True, check=True).stdout


def functions(text: str, ignore_offsets: bool = False) -> dict:
    out, name, body = {}, None, []
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
            continue
        t = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()
        if ignore_offsets:
            t = " ".join(_BANK3.sub(_bank3, _ENCODING.sub("", t)).split())
        if name is None or not t or _HEADER.match(t):
            continue
        body.append(t)
    if name:
        out[name] = body
    return out


def main(old: str, new: str, ignore_offsets: bool = False) -> int:
    a, b = functions(_listing(old), ignore_offsets), functions(_listing(new), ignore_offsets)
    same = [k for k in a if b.get(k) == a[k]]
    diff = [k for k in a if k in b and b[k] != a[k]]
    gone = [k for k in a if k not in b]
    added = [k for k in b if k not in a]
    n_ins = sum(sum(1 for ln in a[k] if ";" in ln) for k in same)
    print(f"{os.path.basename(old)}: {len(a)} functions; identical in {os.path.basename(new)}: {len(same)} "
          f"({n_ins} instructions); differing {len(diff)}; gone {len(gone)}; new {len(added)}")
    for tag, names in (("DIFFERS", diff), ("GONE", gone), ("NEW", added)):
        for k in sorted(names):
            print(f"  {tag} {k}")
    return 1 if diff or gone else 0


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if a != "--ignore-offsets"]
    if len(args) != 2:
        sys.exit(__doc__)
    sys.exit(main(args[0], args[1], "--ignore-offsets" in sys.argv))
