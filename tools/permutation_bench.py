#!/usr/bin/env python3
"""Time pcs_permutation_partial_products (the permutation argument's Zs and partial products) at the benchmark's shape:
80 routed wires x 2^20 rows, 2 challenges, quotient_degree_factor 8 (standard_recursion_config, degree 2^20).

    python tools/permutation_bench.py [--lg-n 20] [--reps 20] [--out results/permutation_bench.json]

Prints one JSON object: the GPU's name and power limit (read in the same run), the device time of one call with device
inputs (CUDA events on the engine's stream after warm-up, median and spread over --reps calls), the same call from pageable
host arrays (host clock around the synchronous call), per-kernel device times from torch.profiler (a separate pass), the CPU
oracle's time on all host cores, and the bytes and field multiplications the shape implies.  Outputs are checked against the
oracle first.  Needs a CUDA device; writes only to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "harness"))

import numpy as np  # noqa: E402

import permutation_oracle as po  # noqa: E402

P = 0xFFFFFFFF00000001
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def counts(R, n, C, D):
    K = -(-R // D)
    Pp = K - 1
    W = C * (1 + Pp)
    mults_rows = n * C * (4 * R + 2 * K + 2 * Pp + 1) + n * -(-C // 4) * (73 + 3 * min(C, 4))
    mults_scan = 3 * n * C
    mults_mul_z = n * C * Pp
    return {
        "algorithmic_read_bytes": 2 * R * n * 8,
        "algorithmic_write_bytes": W * n * 8,
        "engine_bytes": (2 * R * n + C * Pp * n + C * n        # step 1: wires + sigmas in; row-local prefixes, T out
                         + 2 * C * n + C * n                    # scan: T read twice, Z out
                         + C * n + 2 * C * Pp * n) * 8,         # step 3: Z, prefixes read and written
        "num_den_pairs": R * n * C,
        "row_inversions": n * -(-C // 4),
        "field_mults": mults_rows + mults_scan + mults_mul_z,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lg-n", type=int, default=20)
    ap.add_argument("--routed", type=int, default=80)
    ap.add_argument("--challenges", type=int, default=2)
    ap.add_argument("--degree-factor", type=int, default=8)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    if not torch.cuda.is_available():
        sys.exit("permutation_bench needs a CUDA device")
    R, lg_n, C, D = a.routed, a.lg_n, a.challenges, a.degree_factor
    n = 1 << lg_n
    rng = np.random.default_rng(2024)
    wires = rng.integers(0, 1 << 64, (R, n), dtype=np.uint64, endpoint=False)
    sigmas = rng.integers(0, 1 << 64, (R, n), dtype=np.uint64, endpoint=False)
    k_is = p.get_unique_coset_shifts(n, R)
    betas = rng.integers(0, P, C, dtype=np.uint64)
    gammas = rng.integers(0, P, C, dtype=np.uint64)

    ncores = po.use_all_cores()
    t0 = time.perf_counter()
    want = po.prove_order(po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D))
    oracle_s = time.perf_counter() - t0
    W = want.shape[0]

    stream = torch.cuda.current_stream()
    p.init(0, stream.cuda_stream)
    L = _ffi.lib()
    w_dev = torch.from_numpy(wires.view(np.int64)).cuda()
    s_dev = torch.from_numpy(sigmas.view(np.int64)).cuda()
    o_dev = torch.empty((W, n), dtype=torch.int64, device="cuda")
    args = (_ffi.dev_ptr_array(w_dev.data_ptr(), R, n), _ffi.dev_ptr_array(s_dev.data_ptr(), R, n), R, lg_n, _ffi.ptr(k_is),
            _ffi.ptr(betas), _ffi.ptr(gammas), C, D, _ffi.PCS_DEVICE_PTRS, _ffi.dev_ptr_array(o_dev.data_ptr(), W, n))

    def dev_call():
        _ffi.check(L.pcs_permutation_partial_products(*args))

    dev_call()
    assert np.array_equal(o_dev.cpu().numpy().view(np.uint64), want), "device result differs from the oracle"
    for _ in range(a.warmup):
        dev_call()
    ms = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        dev_call()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))

    host_out = np.empty((W, n), dtype=np.uint64)
    host_args = (_ffi.ptr_array(list(wires)), _ffi.ptr_array(list(sigmas)), R, lg_n, _ffi.ptr(k_is), _ffi.ptr(betas),
                 _ffi.ptr(gammas), C, D, 0, _ffi.ptr_array(list(host_out)))
    _ffi.check(L.pcs_permutation_partial_products(*host_args))
    assert np.array_equal(host_out, want), "host-input result differs from the oracle"
    host_ms = []
    for _ in range(max(3, a.reps // 4)):
        t0 = time.perf_counter()
        _ffi.check(L.pcs_permutation_partial_products(*host_args))
        host_ms.append(1e3 * (time.perf_counter() - t0))

    # per-kernel device times, in a pass of its own
    from torch.profiler import ProfilerActivity, profile

    kernels = {}
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                dev_call()
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
            if t and ev.key.startswith(("_ZN", "k_", "void")):
                kernels[ev.key[:90]] = round(t / 5 / 1e3, 4)   # ms per call
    except Exception as e:   # the timed numbers above stand without the breakdown
        kernels = {"error": repr(e)[:200]}

    c = counts(R, n, C, D)
    med = statistics.median(ms)
    res = {
        "gpu": gpu_info(),
        "shape": {"num_routed_wires": R, "lg_n": lg_n, "num_challenges": C, "quotient_degree_factor": D, "outputs": W},
        "device_inputs_ms": {"median": round(med, 4), "min": round(min(ms), 4), "max": round(max(ms), 4), "reps": a.reps},
        "host_inputs_ms": {"median": round(statistics.median(host_ms), 3), "min": round(min(host_ms), 3), "reps": len(host_ms)},
        "kernels_ms_per_call": kernels,
        "cpu_oracle_s": round(oracle_s, 3),
        "cpu_oracle_threads": ncores,
        **c,
        "read_bound_ms": round(c["algorithmic_read_bytes"] / HBM_BYTES_PER_S * 1e3, 4),
        "read_bound_fraction_of_call": round(c["algorithmic_read_bytes"] / HBM_BYTES_PER_S * 1e3 / med, 3),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    p.shutdown()


if __name__ == "__main__":
    main()
