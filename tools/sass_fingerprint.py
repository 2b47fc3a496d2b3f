"""SHA-256 of a library's SASS listing (cuobjdump -sass, instruction text only: no encodings, and the anonymous-namespace
hash that nvcc derives from the source path is masked in function names, so two builds of the same sources compare equal
even at different paths and with different temporary-file names).  Used to show that the in-tree libpcs.so is, instruction
for instruction, the binary a GPU run tested (profiles/r02_forms.md).

    python tools/sass_fingerprint.py [path/to/libpcs.so]
"""
import hashlib
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fingerprint(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    h, n = hashlib.sha256(), 0
    for line in out.split("\n"):
        m = re.search(r"Function : (\S+)", line)
        if m:
            h.update(("F " + re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1)) + "\n").encode())
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,6})\*/\s+(.*?);", line)
        if m:
            h.update((m.group(1) + " " + " ".join(m.group(2).split()) + "\n").encode())
            n += 1
    return h.hexdigest(), n


if __name__ == "__main__":
    lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "plonky2_demo_b200", "libpcs.so")
    fp, n = fingerprint(lib)
    print(f"{fp}  {n} instructions  {os.path.relpath(lib, ROOT)}")
