#!/usr/bin/env python3
"""Time pcs_quotient_polys (prove()'s quotient chunks without the gate constraints) at the standard shape -- degree 2^20,
80 routed wires, 2 challenges, quotient_degree_factor 8, rate 3 (standard_recursion_config) -- and at the m = 64 demo
shape (degree 2^15).

    python tools/quotient_bench.py [--lg-n 20,15] [--reps 20] [--out results/quotient_bench.json]

Prints one JSON object: the GPU's name and power limit (read in the same run) and, per shape, the device time of one call
with device outputs (CUDA events on the engine's stream after warm-up, median and spread over --reps calls), the same call
into pageable host arrays (host clock around the synchronous call), per-kernel device times from torch.profiler (a separate
pass; k_quotient_points is the point kernel), the CPU oracle's time for the same step on all host cores, and the bytes and
field multiplications the shape implies.  Outputs are checked against the oracle first.  Needs a CUDA device; writes only to
--out."""
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

import quotient_oracle as qo  # noqa: E402

P = 0xFFFFFFFF00000001
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def counts(R, n, C, D):
    K = -(-R // D)
    Pp = K - 1
    M = n << (D - 1).bit_length()
    per_point = (4 * R * C            # beta k_j x, beta sigma_j and the two running products per wire and challenge
                 + K * C * (2 + C)    # prev * N - next * D per chunk, one Horner step per alpha
                 + C * (1 + C)        # L_0 (Z - 1) and its alpha powers
                 + C * C + 2 * C + 2 + 4)   # the blocks put together, Z_H^-1, L_0, x, Montgomery's trick
    return {
        "points": M,
        # wires, sigmas, Zs and partial products at every point, plus Z(g x): the bytes the point kernel must read
        "point_kernel_read_bytes": (2 * R + C * (1 + Pp) + C) * M * 8,
        "point_kernel_write_bytes": C * M * 8,
        "field_mults_per_point": per_point + 72 // 4,   # one inversion (72 multiplications) per 4 points
        "field_mults": (per_point + 72 // 4) * M,
    }


def bench_shape(L, p, _ffi, torch, stream, lg_n, R, C, D, rate_bits, reps, warmup):
    import oracle

    n = 1 << lg_n
    K = -(-R // D)
    rng = np.random.default_rng(lg_n)
    coeffs = [rng.integers(0, P, (w, n), dtype=np.uint64) for w in (R, R, C * K)]   # sigmas, wires, Zs + partial products
    k_is = p.get_unique_coset_shifts(n, R)
    betas, gammas, alphas = (rng.integers(0, P, C, dtype=np.uint64) for _ in range(3))

    oracle.use_all_cores()
    ncores = qo.use_all_cores()
    lde = [oracle.coset_lde(c, rate_bits) for c in coeffs]
    t0 = time.perf_counter()
    want = qo.quotient_poly_chunks(qo.compute_quotient_polys(*lde, rate_bits, 0, R, k_is, betas, gammas, alphas, D), n, D)
    oracle_s = time.perf_counter() - t0
    del lde

    batches = [p.PolynomialBatch.from_coeffs(c, rate_bits, False, 4) for c in coeffs]
    W = C * D
    o_dev = torch.empty((W, n), dtype=torch.int64, device="cuda")
    scal = (0, R, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas), _ffi.ptr(alphas), C, D, None)
    hs = tuple(b._h for b in batches)

    def dev_call():
        _ffi.check(L.pcs_quotient_polys(*hs, *scal, _ffi.PCS_DEVICE_PTRS, _ffi.dev_ptr_array(o_dev.data_ptr(), W, n)))

    dev_call()
    assert np.array_equal(o_dev.cpu().numpy().view(np.uint64), want), "device result differs from the oracle"
    for _ in range(warmup):
        dev_call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        dev_call()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))

    host_out = np.empty((W, n), dtype=np.uint64)
    host_args = (*hs, *scal, 0, _ffi.ptr_array(list(host_out)))
    _ffi.check(L.pcs_quotient_polys(*host_args))
    assert np.array_equal(host_out, want), "host-output result differs from the oracle"
    host_ms = []
    for _ in range(max(3, reps // 4)):
        t0 = time.perf_counter()
        _ffi.check(L.pcs_quotient_polys(*host_args))
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
            if t and ev.key.startswith(("_ZN", "k_", "void", "Memcpy", "Memset")):
                kernels[ev.key[:90]] = round(t / 5 / 1e3, 4)   # ms per call
    except Exception as e:   # the timed numbers above stand without the breakdown
        kernels = {"error": repr(e)[:200]}
    point_ms = sum(v for k, v in kernels.items() if isinstance(v, float) and "k_quotient_points" in k)
    for b in batches:   # now, not at garbage collection after pcs_shutdown
        b.free()

    c = counts(R, n, C, D)
    med = statistics.median(ms)
    res = {
        "shape": {"num_routed_wires": R, "lg_n": lg_n, "num_challenges": C, "quotient_degree_factor": D, "rate_bits": rate_bits,
                  "outputs": W},
        "device_outputs_ms": {"median": round(med, 4), "min": round(min(ms), 4), "max": round(max(ms), 4), "reps": reps},
        "host_outputs_ms": {"median": round(statistics.median(host_ms), 3), "min": round(min(host_ms), 3), "reps": len(host_ms)},
        "kernels_ms_per_call": kernels,
        "point_kernel_ms": round(point_ms, 4),
        "cpu_oracle_s": round(oracle_s, 3),
        "cpu_oracle_threads": ncores,
        **c,
        "point_kernel_read_bound_ms": round(c["point_kernel_read_bytes"] / HBM_BYTES_PER_S * 1e3, 4),
    }
    if point_ms:
        res["point_kernel_read_tb_per_s"] = round(c["point_kernel_read_bytes"] / (point_ms * 1e-3) / 1e12, 3)
        res["point_kernel_gmults_per_s"] = round(c["field_mults"] / (point_ms * 1e-3) / 1e9, 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lg-n", default="20,15")
    ap.add_argument("--routed", type=int, default=80)
    ap.add_argument("--challenges", type=int, default=2)
    ap.add_argument("--degree-factor", type=int, default=8)
    ap.add_argument("--rate-bits", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    if not torch.cuda.is_available():
        sys.exit("quotient_bench needs a CUDA device")
    stream = torch.cuda.current_stream()
    p.init(0, stream.cuda_stream)
    L = _ffi.lib()
    res = {"gpu": gpu_info(), "shapes": []}
    for lg_n in (int(v) for v in a.lg_n.split(",")):
        res["shapes"].append(bench_shape(L, p, _ffi, torch, stream, lg_n, a.routed, a.challenges, a.degree_factor, a.rate_bits,
                                         a.reps, a.warmup))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    p.shutdown()


if __name__ == "__main__":
    main()
