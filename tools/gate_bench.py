#!/usr/bin/env python3
"""Time pcs_gate_constraint_terms (the gate-constraint tail of prove()'s quotient step) with the matmul demo's gate set and
grouping ([NoopGate, ConstantGate(2), PublicInputGate, ArithmeticGate(20)] and [PoseidonGate]: 2 selectors, 4 constants, 135
wires), at the standard shape -- degree 2^20, 2 challenges, quotient_degree_factor 8, rate 3 -- and at the m = 64 demo shape
(degree 2^15).

    python tools/gate_bench.py [--lg-n 20,15] [--reps 20] [--out results/gate_bench.json]

Prints one JSON object: the GPU's name and power limit (read in the same run) and, per shape, the device time of one call with
device outputs (CUDA events on the engine's stream after warm-up, median and spread over --reps calls), per-kernel device times
from torch.profiler (a separate pass; k_gate_points is the point kernel), the same call into pageable host arrays (host clock
around the synchronous call), the CPU oracle's time on 16 threads, and the whole quotient step -- gate terms + pcs_quotient_polys
-- on the device against the host path a caller without this entry point takes: export the wires and constants batches' LDE rows
(pcs_batch_lde_natural), evaluate the gates on the CPU (the oracle), and pass the tail to pcs_quotient_polys from the host.  The
bytes and field multiplications the shape implies are computed from it.  Outputs are checked against the oracle first.  Needs a
CUDA device; writes only to --out."""
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

import gate_oracle as go  # noqa: E402

P = 0xFFFFFFFF00000001
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
GATES = [(go.NOOP, 0, 0), (go.CONSTANT, 2, 0), (go.PUBLIC_INPUT, 0, 0), (go.ARITHMETIC, 20, 0), (go.POSEIDON, 0, 1)]
GROUPS = [(0, 4), (4, 5)]
NUM_CONSTANTS, WIRES, ROUTED = 4, 135, 80


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def counts(n, C, D):
    M = n << (D - 1).bit_length()
    poseidon = 118 * 4 + 1 + 4 + 123 * C   # S-boxes (4 multiplications each), swap, deltas, one per constraint and alpha
    arithmetic = 20 * 3 + 20 * C
    others = 2 * C + 4 * C                 # ConstantGate, PublicInputGate
    filters = 3 * 4 + 1 + 4 * C            # group [0, 4): 3 factors + UNUSED_SELECTOR for 3 gates; PoseidonGate: 1; times acc
    per_point = poseidon + arithmetic + others + filters
    return {
        "points": M,
        "point_kernel_read_bytes": (WIRES + NUM_CONSTANTS) * M * 8,   # every wire column and the 4 constant columns
        "point_kernel_write_bytes": C * M * 8,
        "field_mults_per_point": per_point,
        "field_mults": per_point * M,
        "mds_layers_per_point": 30,   # FP64 add/shift network, no field multiplications
    }


def bench_shape(L, p, _ffi, torch, stream, lg_n, C, D, rate_bits, reps, warmup):
    import oracle

    n = 1 << lg_n
    M = n << (D - 1).bit_length()
    K = -(-ROUTED // D)
    rng = np.random.default_rng(lg_n)
    cs = rng.integers(0, P, (NUM_CONSTANTS + ROUTED, n), dtype=np.uint64)
    wires = rng.integers(0, P, (WIRES, n), dtype=np.uint64)
    zs = rng.integers(0, P, (C * K, n), dtype=np.uint64)
    pih, alphas, betas, gammas = (rng.integers(0, P, s, dtype=np.uint64) for s in (4, C, C, C))
    k_is = p.get_unique_coset_shifts(n, ROUTED)
    gates = np.ascontiguousarray(np.array(GATES, dtype=np.uint32))
    groups = np.ascontiguousarray(np.array(GROUPS, dtype=np.uintp))

    batches = [p.PolynomialBatch.from_coeffs(c, rate_bits, False, 4) for c in (cs, wires, zs)]
    hs = tuple(b._h for b in batches)
    gt_dev = torch.empty((C, M), dtype=torch.int64, device="cuda")
    q_dev = torch.empty((C * D, n), dtype=torch.int64, device="cuda")
    gt_table = _ffi.dev_ptr_array(gt_dev.data_ptr(), C, M)

    def gate_call(flags, outs):
        _ffi.check(L.pcs_gate_constraint_terms(hs[0], hs[1], gates.ctypes.data_as(_ffi.C.POINTER(_ffi.C.c_uint32)), len(GATES),
                                               groups.ctypes.data_as(_ffi.C.POINTER(_ffi.sz)), len(GROUPS), 0, NUM_CONSTANTS,
                                               _ffi.ptr(pih), _ffi.ptr(alphas), C, D, flags, outs))

    q_host = np.empty((C * D, n), dtype=np.uint64)
    q_dev_table, q_host_table = _ffi.dev_ptr_array(q_dev.data_ptr(), C * D, n), _ffi.ptr_array(list(q_host))

    def quotient_call(tail, flags, outs):   # flags cover the tail and the outputs alike
        _ffi.check(L.pcs_quotient_polys(*hs, NUM_CONSTANTS, ROUTED, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas),
                                        _ffi.ptr(alphas), C, D, tail, flags, outs))

    def dev_call():
        gate_call(_ffi.PCS_DEVICE_PTRS, gt_table)

    def timed(fn, count):
        ms = []
        for _ in range(count):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return ms

    # the host path's first two steps: export the LDE rows of both batches, evaluate the gates on the CPU
    t0 = time.perf_counter()
    for b in batches[:2]:
        rows = np.empty((M, b.n_polys), dtype=np.uint64)
        _ffi.check(L.pcs_batch_lde_natural(b._h, 0, 1 << (rate_bits - (D - 1).bit_length()), M, _ffi.ptr(rows)))
        del rows
    export_s = time.perf_counter() - t0
    oracle.use_all_cores()
    go.set_num_threads(16)
    lde = [oracle.coset_lde(cs[:NUM_CONSTANTS], rate_bits), oracle.coset_lde(wires, rate_bits)]
    t0 = time.perf_counter()
    want = go.gate_terms(*lde, rate_bits, GATES, GROUPS, NUM_CONSTANTS, pih, alphas, D)
    oracle_s = time.perf_counter() - t0
    del lde

    dev_call()
    assert np.array_equal(gt_dev.cpu().numpy().view(np.uint64), want), "device result differs from the oracle"
    for _ in range(warmup):
        dev_call()
    ms = timed(dev_call, reps)

    host_out = np.empty((C, M), dtype=np.uint64)
    host_table = _ffi.ptr_array(list(host_out))
    gate_call(0, host_table)
    assert np.array_equal(host_out, want), "host-output result differs from the oracle"
    host_ms = []
    for _ in range(max(3, reps // 4)):
        t0 = time.perf_counter()
        gate_call(0, host_table)
        host_ms.append(1e3 * (time.perf_counter() - t0))

    # the whole quotient step on the device: gate terms into a device tail, pcs_quotient_polys from it
    def step_dev():
        dev_call()
        quotient_call(gt_table, _ffi.PCS_DEVICE_PTRS, q_dev_table)

    # the host path's last step: the host tail into pcs_quotient_polys, host outputs
    host_tail = _ffi.ptr_array(list(want))
    step_dev()
    quotient_call(host_tail, 0, q_host_table)
    assert np.array_equal(q_dev.cpu().numpy().view(np.uint64), q_host), "host and device tails give other chunks"
    for _ in range(warmup):
        step_dev()
    step_ms = timed(step_dev, reps)
    q_host_ms = []
    for _ in range(max(3, reps // 4)):
        t0 = time.perf_counter()
        quotient_call(host_tail, 0, q_host_table)
        q_host_ms.append(1e3 * (time.perf_counter() - t0))

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
    point_ms = sum(v for k, v in kernels.items() if isinstance(v, float) and "k_gate_points" in k)
    for b in batches:   # now, not at garbage collection after pcs_shutdown
        b.free()

    c = counts(n, C, D)
    med = statistics.median(ms)
    host_path_ms = 1e3 * (export_s + oracle_s) + statistics.median(q_host_ms)
    res = {
        "shape": {"wires": WIRES, "num_constants": NUM_CONSTANTS, "num_routed_wires": ROUTED, "lg_n": lg_n, "num_challenges": C,
                  "quotient_degree_factor": D, "rate_bits": rate_bits},
        "device_outputs_ms": {"median": round(med, 4), "min": round(min(ms), 4), "max": round(max(ms), 4), "reps": reps},
        "host_outputs_ms": {"median": round(statistics.median(host_ms), 3), "min": round(min(host_ms), 3), "reps": len(host_ms)},
        "kernels_ms_per_call": kernels,
        "point_kernel_ms": round(point_ms, 4),
        "cpu_oracle_s": round(oracle_s, 3),
        "cpu_oracle_threads": 16,
        "quotient_step_device_ms": {"median": round(statistics.median(step_ms), 3), "min": round(min(step_ms), 3), "reps": reps},
        "quotient_step_host_path_ms": {"total": round(host_path_ms, 1), "lde_rows_export_ms": round(1e3 * export_s, 1),
                                       "cpu_gate_terms_ms": round(1e3 * oracle_s, 1),
                                       "quotient_polys_host_tail_ms": round(statistics.median(q_host_ms), 3)},
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
        sys.exit("gate_bench needs a CUDA device")
    stream = torch.cuda.Stream()   # the engine's stream too: events and copies are ordered behind its asynchronous work
    torch.cuda.set_stream(stream)
    p.init(0, stream.cuda_stream)
    L = _ffi.lib()
    res = {"gpu": gpu_info(), "shapes": []}
    for lg_n in (int(v) for v in a.lg_n.split(",")):
        res["shapes"].append(bench_shape(L, p, _ffi, torch, stream, lg_n, a.challenges, a.degree_factor, a.rate_bits, a.reps,
                                         a.warmup))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    p.shutdown()


if __name__ == "__main__":
    main()
