"""Compare the device code of two builds of libsart.so function by function.

    python tools/compare_sass.py OLD.so NEW.so

Runs `cuobjdump -sass` on both libraries, splits each listing at its `Function :` headers and reports the functions
only one build has and the functions present in both whose SASS differs. Exits 1 if any function present in both builds
differs. Two clean builds of the same commit give identical listings, so a difference is a real change in device code.
"""
from __future__ import annotations

import os
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def functions(lib: str) -> dict[str, str]:
    text = subprocess.run([CUOBJDUMP, "-sass", lib], check=True, capture_output=True, text=True).stdout
    out: dict[str, str] = {}
    name, body = None, []
    for line in text.splitlines():
        if line.strip().startswith("Function :"):
            name, body = line.split(":", 1)[1].strip(), []
        elif name is not None and line.strip().startswith(".........."):   # end of the function's listing
            out[name] = "\n".join(body)
            name = None
        elif name is not None:
            body.append(line)
    return out


def main(argv: list[str]) -> int:
    if len(argv) != 3:
        print(__doc__.strip())
        return 2
    old, new = functions(argv[1]), functions(argv[2])
    gone, added = sorted(old.keys() - new.keys()), sorted(new.keys() - old.keys())
    changed = sorted(k for k in old.keys() & new.keys() if old[k] != new[k])
    print(f"{len(old)} functions before, {len(new)} after; {len(old.keys() & new.keys()) - len(changed)} identical")
    for title, names in (("only before", gone), ("only after", added), ("different", changed)):
        for n in names:
            print(f"{title}: {n}")
    return 1 if changed else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
