"""ORACLE -- test infrastructure, NOT the product: the build shared by the ctypes front-ends of the C oracles in this directory.
A library is compiled on first use with gcc into a per-user temporary directory keyed by the hash of its source and headers, so
a read-only tree works too."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_DIR = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "oracle")   # gl64.h, poseidon_constants.h
u64p = C.POINTER(C.c_uint64)


def build(name, headers=("gl64.h",)):
    """Compile <name>.c of this directory (if needed) against the oracle's `headers`; return the shared library's path."""
    src = os.path.join(_HERE, name + ".c")
    h = hashlib.sha256()
    for f in (src,) + tuple(os.path.join(_ORACLE_DIR, x) for x in headers):
        with open(f, "rb") as fh:
            h.update(fh.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"pcs_{name}_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"lib{name}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-Wall", "-Wextra",
                               "-std=gnu11", "-shared", "-I", _ORACLE_DIR, "-o", tmp, src])
        os.replace(tmp, so)
    return so


def use_all_cores(set_num_threads):
    """set_num_threads(the number of CPUs this process may run on); returns that number"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    set_num_threads(n)
    return n


def u64(a):
    return np.ascontiguousarray(a, dtype=np.uint64)
