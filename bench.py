#!/usr/bin/env python3
"""Headline benchmark: LDE + Merkle commit throughput (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one PolynomialBatch::from_coeffs commit (plonky2/src/fri/oracle.rs:68-98) of
135 polynomials of degree 2^20 at rate_bits 3, cap_height 4 (BASELINE.json configs[3]):
batched Goldilocks coset LDE -> Poseidon leaf hashing -> Merkle levels up to the cap.
`elems` = LDE output field elements committed = W * N = 135 * 2^23 per commit (SURVEY 8d).

  value : device-resident throughput (coefficients already in HBM), CUDA events on the engine's stream
  e2e   : the same commit through the C ABI with HOST buffers: pinned host coefficients -> H2D ->
          commit -> D2H of the Merkle cap, every step, inside the timed region
  roofline     : dominant kernel (Poseidon leaf hashing) against the measured HBM peak
  cpu_baseline : the CPU oracle (C/OpenMP port of the reference algorithm) on a bounded sample

N > 1 (torchrun, one rank per GPU): the SAME commitment sharded over the N GPUs (BASELINE.json configs[3]:
"... at 1/2/4/8 GPUs") -> strong scaling.  Rank r starts with its block of the 135 polynomials in HBM; a step is
NCCL all-gather of the coefficients -> LDE of the rank's coset blocks (= a contiguous leaf range) -> leaf hashing
-> the rank's cap subtrees -> NCCL all-gather of the cap (plonky2_demo_b200/sharded.py).
value = W*N elems / max-over-ranks time.

--impl reference times the CPU port of the reference (oracle/) with all host threads on a bounded
sample of the same workload; rank 0 only.

--dump-outputs DIR writes what the last timed commit computed, so that two builds can be compared output for output
(the inputs are the same seeded polynomials on every run): DIR/cap.npy [2^cap_height][4][2], and for a fixed, seeded
sample of leaves DIR/leaf_indices.npy [k], DIR/leaves.npy [k][width][2] (the LDE rows) and DIR/merkle_paths.npy
[k][log2 N - cap_height][4][2] (MerkleTree::prove).  Field elements are 64-bit, so every one is stored as its low and
high 32-bit halves (last axis), which float64 holds exactly; the files stay below 64 MB in all.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "lde_merkle_commit_elems_per_s"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE k_hash_cols launch, from the `ncu --set full` capture of this very
# command on the shipped build (tools/gpu_profile.sh writes profiles/leafhash_traffic.json next to the summary it comes from)
def ncu_traffic(width, lg_d, rate_bits, n_gpus):
    p = os.path.join(ROOT, "profiles", "leafhash_traffic.json")
    try:
        with open(p) as f:
            t = json.load(f)
    except (OSError, ValueError):
        return None, "no capture"
    key = f"{width}x2^{lg_d}_r{rate_bits}_g{n_gpus}"
    e = t.get(key)
    if not e:
        return None, "no capture for this shape"
    return int(e["dram_bytes_read"]) + int(e["dram_bytes_write"]), e.get("source", "profiles/leafhash_traffic.json")


# thread-instructions per Poseidon permutation of the shipped k_hash_cols (ncu smsp__inst_executed x 32 / permutations, or the
# static SASS count of its loop bodies when no capture of this build exists): profiles/leafhash_instr.json
def leafhash_instr():
    try:
        with open(os.path.join(ROOT, "profiles", "leafhash_instr.json")) as f:
            e = json.load(f)
        return float(e["thread_instr_per_permutation"]), e.get("source", "profiles/leafhash_instr.json")
    except (OSError, ValueError, KeyError):
        return 17080.0, "profiles/r02_leafhash.md: 7.611e10 warp-instructions x 32 / (17 x 2^23) (round-2 build)"


UNIT = "elems/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=135)
    ap.add_argument("--lg-d", type=int, default=20)
    ap.add_argument("--rate-bits", type=int, default=3)
    ap.add_argument("--cap-height", type=int, default=4)
    ap.add_argument("--cpu-sample-lg-d", type=int, default=16, help="degree_log of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--reference-full-size", default="auto", choices=["auto", "on", "off"],
                    help="--impl reference: also run the full 2^lg_d configuration on the CPU (auto: when it fits the budgets)")
    ap.add_argument("--reference-budget-s", type=float, default=150.0)
    ap.add_argument("--large-commit", default="auto", choices=["auto", "on", "off"],
                    help="N = 8: add BASELINE configs[4], one 135 x 2^24 commitment sharded over the box, with sampled-leaf parity")
    ap.add_argument("--no-from-values", action="store_true", help="skip the from_values timing at the headline size")
    ap.add_argument("--no-multi-in-process", action="store_true", help="N > 1: skip the pcs_multi_* (one process, N GPUs) timing")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fri", action="store_true", help="skip the opening-proof (FRI) timings")
    ap.add_argument("--chunks", default="3",
                    help="N > 1: polynomial groups of the streaming exchange in the device-resident arm: a count (first group 8 "
                         "polynomials, the rest equal) or host:<rho> (1 = one all-gather, then the LDE)")
    ap.add_argument("--e2e-chunks", default="auto",
                    help="N > 1: groups of the END-TO-END arm, where every group also crosses PCIe first.  auto = host:<rho> with "
                         "rho = transfer / compute time per polynomial (0.75 at N >= 4 where the host side saturates, 0.4 at N = 2): "
                         "geometrically growing groups, only the first 8-polynomial transfer is exposed")
    ap.add_argument("--exchange", default="auto", choices=["auto", "allgather", "peer", "alltoall"],
                    help="N > 1: how coefficient blocks reach the other ranks (plonky2_demo_b200/sharded.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed commit computed to DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def workload_name(a):
    return f"PolynomialBatch::from_coeffs commit: {a.width} polys x 2^{a.lg_d}, rate_bits {a.rate_bits}, Poseidon MerkleTree cap_height {a.cap_height}"


def bench_config(a):
    """`config` of the JSON line: identical for both arms (the driver compares them)."""
    return {"workload": workload_name(a), "elems_per_step": a.width * (1 << (a.lg_d + a.rate_bits))}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference's CPU path) on a bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_commit_once(width, lg_d, rate_bits, cap_height, keep=False):
    import oracle
    from helpers import seeded_polys

    coeffs = seeded_polys(width, 1 << lg_d)
    t0 = time.perf_counter()
    out = oracle.commit_from_coeffs(coeffs, rate_bits, cap_height)
    dt = time.perf_counter() - t0
    cap = out["cap"].copy()
    del out
    return dt, cap


DUMP_BUDGET_BYTES = 48 << 20


def dump_sample(n_leaves, leaf_len, depth):
    """--dump-outputs: the same sorted leaf indices on every run, as many as fit the budget (4096 at most)."""
    per_leaf = 8 + 16 * (leaf_len + 4 * depth)
    k = max(1, min(n_leaves, 4096, DUMP_BUDGET_BYTES // per_leaf))
    return np.sort(np.random.default_rng(0x5EED).choice(n_leaves, size=k, replace=False)).astype(np.uint64)


def write_outputs(out_dir, leaf_indices, field_arrays):
    """leaf_indices as float64 (exact below 2^53); field elements as float64 [..., 2] = (low, high) 32-bit halves."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "leaf_indices.npy"), leaf_indices.astype(np.float64))
    for name, a in field_arrays.items():
        a = np.asarray(a, dtype=np.uint64)
        np.save(os.path.join(out_dir, name + ".npy"),
                np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64))


def _mem_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def cpu_baseline(a):
    import oracle

    cores = oracle.use_all_cores()   # torchrun exports OMP_NUM_THREADS=1: the reference's rayon pool uses every core
    lg = min(a.cpu_sample_lg_d, a.lg_d)
    dt, _ = cpu_commit_once(a.width, lg, a.rate_bits, a.cap_height)
    elems = a.width * (1 << (lg + a.rate_bits))
    return {
        "value": elems / dt,
        "unit": UNIT,
        "cores": cores,
        "kind": "port",
        "sample": f"one from_coeffs commit of {a.width} x 2^{lg} (rate_bits {a.rate_bits}, cap_height {a.cap_height}), "
                  f"{dt:.2f} s wall on {cores} OpenMP threads; C port of the reference CPU algorithm (oracle/oracle.c)",
    }


def run_reference(a):
    """--impl reference: the CPU port of the reference path on ALL host cores (whatever OMP_NUM_THREADS torchrun exported).
    The K timed steps are K - 1 bounded samples (135 x 2^cpu_sample_lg_d) and ONE commit of the full configuration (all K full-size
    when K <= 3); the full-size step is dropped -- and says so -- when it would not fit the time / memory budget.
    value = elements committed in the timed region / its duration.  Rank 0 only; the other ranks exit at once."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle

    cores = oracle.use_all_cores()
    lg = min(a.cpu_sample_lg_d, a.lg_d)
    for _ in range(min(a.warmup, 2)):
        cpu_commit_once(a.width, lg, a.rate_bits, a.cap_height)
    elems_s = a.width * (1 << (lg + a.rate_bits))
    elems_f = a.width * (1 << (a.lg_d + a.rate_bits))
    # probe: one sample step decides whether the full configuration fits
    probe, _ = cpu_commit_once(a.width, lg, a.rate_bits, a.cap_height)
    n_full, skipped = 0, None
    if lg < a.lg_d and a.reference_full_size != "off":
        want = a.steps if a.steps <= 3 else 1
        predicted = probe * (1 << (a.lg_d - lg)) * 1.4            # cache effects make the big case slower per element
        need = int(elems_f * 8 * 2.6)                              # LDE + transposed leaves + coefficients + digests
        avail = _mem_available_bytes()
        if a.reference_full_size == "on" or (predicted * want <= a.reference_budget_s and avail >= need):
            n_full = want
        else:
            skipped = (f"predicted {predicted * want:.0f} s (budget {a.reference_budget_s} s), needs {need >> 30} GiB of host memory "
                       f"({avail >> 30} GiB available)")
    elif lg == a.lg_d:
        n_full = a.steps
    sample_t, full_t = [], []
    for k in range(a.steps):
        if k >= a.steps - n_full and lg < a.lg_d:
            dt, _ = cpu_commit_once(a.width, a.lg_d, a.rate_bits, a.cap_height)
            full_t.append(dt)
        else:
            dt, _ = cpu_commit_once(a.width, lg, a.rate_bits, a.cap_height)
            (full_t if lg == a.lg_d else sample_t).append(dt)
    total = sum(sample_t) + sum(full_t)
    elems = elems_s * len(sample_t) + elems_f * len(full_t)
    value = elems / total
    sample = (f"{a.steps} timed steps on {cores} OpenMP threads: {len(sample_t)} bounded samples (one from_coeffs commit of {a.width} x 2^{lg} each"
              f"{', %.2f s' % (sum(sample_t) / len(sample_t)) if sample_t else ''}) and {len(full_t)} commit(s) of the full {a.width} x 2^{a.lg_d} "
              f"configuration{' (%.1f s each)' % (sum(full_t) / len(full_t)) if full_t else ''}; elems/s = elements committed / time"
              + (f"; full-size step skipped: {skipped}" if skipped else ""))
    print(json.dumps({
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * total / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64 (Goldilocks field, integer)", "data": "synthetic",
        "config": bench_config(a),
        "measured_on_full_config": bool(full_t),
        "sample_value": (elems_s * len(sample_t) / sum(sample_t)) if sample_t else None,
        "full_size": ({"runs": len(full_t), "s_per_commit": full_t, "value": elems_f * len(full_t) / sum(full_t), "unit": UNIT} if full_t
                      else {"skipped": skipped}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.samples:
            if ts < t0 or ts > t1 + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def fri_opening_bench(pcs, w, lg_d, r, cap_h, dev_ptrs, steps, peak_gbs):
    """SURVEY 8f N2/N3 at the headline shape: the opening proof over ONE committed batch of w polynomials of degree
    2^lg_d (coefficients kept on the device): every polynomial opened at zeta, the first 20 also at g*zeta (the shape of
    the reference's instance, circuit_data.rs:461-481), standard_recursion_config FRI parameters.  Times are CUDA events
    on the engine's stream around the public calls (each ends with its own small D2H copy)."""
    import torch
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200 import fri_prover as fp

    L = _ffi.lib()
    d = 1 << lg_d
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(dev_ptrs, w, lg_d, r, cap_h, None, 0, _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS,
                                        None, C.byref(h)))
    b = pcs.PolynomialBatch()
    b._h, b._coeffs_host = h, []
    b.degree_log, b.rate_bits, b.blinding, b.cap_height = lg_d, r, False, cap_h
    b.n_polys, b.salt_w, b.n_leaves = w, 0, d << r
    b.n_digests = 2 * ((d << r) - (1 << cap_h))
    cap = np.empty((1 << cap_h, 4), dtype=np.uint64)
    _ffi.check(L.pcs_batch_cap(h, _ffi.ptr(cap)))
    b._cap = cap
    from plonky2_demo_b200.fri import _DeviceMerkleTree
    b.merkle_tree = _DeviceMerkleTree(b)

    stream = torch.cuda.current_stream()

    def timed(fn, reps):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(reps):
            out = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, out

    zeta = (0x0123456789ABCDEF % fp.P, 0x0FEDCBA987654321 % fp.P)
    g = fp.primitive_root_of_unity(lg_d)
    zeta_next = fp.ext_mul((g, 0), zeta)
    n_next = min(20, w)
    inst = fp.FriInstanceInfo(
        oracles=[fp.FriOracleInfo(w, False)],
        batches=[fp.FriBatchInfo(zeta, fp.FriPolynomialInfo.from_range(0, range(w))),
                 fp.FriBatchInfo(zeta_next, fp.FriPolynomialInfo.from_range(0, range(n_next)))])
    alpha = (0x1111111122222222 % fp.P, 0x3333333344444444 % fp.P)

    eval_ms, opened = timed(lambda: fp.eval_commitment(zeta, b), steps)

    def fin():
        p = fp.final_poly(inst, [b], alpha)
        p.free()
    fin_ms, _ = timed(fin, steps)

    cfg = pcs.CircuitConfig.standard_recursion_config().fri_config
    cfg = pcs.FriConfig(r, cap_h, cfg.proof_of_work_bits, cfg.reduction_strategy, cfg.num_query_rounds)
    params = cfg.fri_params(lg_d, False)

    def prove():
        ch = fp.Challenger()
        ch.observe_cap(b.merkle_tree.cap)
        ch.observe_extension_elements([(int(x), int(y)) for x, y in opened[:8]])
        return fp.prove_openings(inst, [b], ch, params)
    prove_ms, proof = timed(prove, max(1, steps // 2))
    eval_bytes = w * d * 8
    fin_bytes = (w + n_next) * d * 8 + 2 * (2 * d * 16 * 3)   # coefficients once per batch + the extension-poly passes
    out = {
        "workload": f"opening proof over {w} polys x 2^{lg_d} (all at zeta, {n_next} at g*zeta), rate_bits {r}, "
                    f"arities {params.reduction_arity_bits}, {cfg.num_query_rounds} queries, {cfg.proof_of_work_bits} PoW bits",
        "eval_commitment": {"ms": eval_ms, "algorithmic_bytes": eval_bytes, "GBps": eval_bytes / (eval_ms * 1e-3) / 1e9,
                            "frac_hbm": eval_bytes / (eval_ms * 1e-3) / 1e9 / peak_gbs},
        "final_poly": {"ms": fin_ms, "algorithmic_bytes": fin_bytes, "GBps": fin_bytes / (fin_ms * 1e-3) / 1e9,
                       "frac_hbm": fin_bytes / (fin_ms * 1e-3) / 1e9 / peak_gbs},
        "prove_openings": {"ms": prove_ms, "final_poly_len": int(proof.final_poly.shape[0]),
                           "commit_phase_trees": len(proof.commit_phase_merkle_caps),
                           "note": "host transcript (Challenger) + device kernels; includes PoW grinding and 28 query rounds"},
    }
    b.free()
    return out


def multi_in_process_bench(a, world, cap_expected):
    """pcs_multi_commit_from_coeffs over `world` GPUs from this ONE process (the other ranks idle at a barrier): host arm =
    pinned host coefficients -> cap on host (each device copies its share over its own PCIe link); device arm = coefficients
    resident, spread round-robin over the GPUs, read in place over NVLink.  Wall-clock around the synchronous calls."""
    import torch

    from helpers import splitmix64_stream
    from plonky2_demo_b200 import _ffi

    L = _ffi.lib()
    w, lg_d, r, cap_h = a.width, a.lg_d, a.rate_bits, a.cap_height
    d = 1 << lg_d
    _ffi.check(L.pcs_multi_init(None, world))
    full = torch.empty((w, d), dtype=torch.int64, pin_memory=True)
    fn = full.numpy().view(np.uint64)
    for j in range(w):
        fn[j] = splitmix64_stream(0x5EED0000 + j, d)
    hp = _ffi.ptr_array([fn[j] for j in range(w)])
    cap = np.empty((1 << cap_h, 4), dtype=np.uint64)
    res = {"devices": world}

    def run(ptrs, flags, reps):
        ts = []
        for _ in range(reps):
            h = C.c_void_p()
            t0 = time.perf_counter()
            _ffi.check(L.pcs_multi_commit_from_coeffs(ptrs, w, lg_d, r, cap_h, None, 0, flags, _ffi.ptr(cap), C.byref(h)))
            ts.append(1e3 * (time.perf_counter() - t0))
            ms5 = (C.c_float * 5)()
            _ffi.check(L.pcs_multi_batch_timings(h, ms5))
            L.pcs_multi_batch_free(h)
        return ts, list(ms5)

    ts, ph = run(hp, 0, 2 + a.steps)
    res["host_inputs"] = {"ms": float(np.median(ts[2:])), "ms_min": float(min(ts[2:])), "cap_equal": bool(np.array_equal(cap, cap_expected)),
                          "phase_ms_max_over_devices": {"FFT + blinding (incl. waits for H2D)": ph[1], "leaf hashing": ph[3], "node levels": ph[4]}}
    tens = [torch.from_numpy(fn[j].view(np.int64)).to(f"cuda:{j % world}") for j in range(w)]
    for g in range(world):
        torch.cuda.synchronize(g)
    dp = (_ffi.u64p * w)(*[C.cast(C.c_void_p(t.data_ptr()), _ffi.u64p) for t in tens])
    ts, ph = run(dp, _ffi.PCS_DEVICE_PTRS, 2 + a.steps)
    res["device_inputs"] = {"ms": float(np.median(ts[2:])), "ms_min": float(min(ts[2:])), "cap_equal": bool(np.array_equal(cap, cap_expected)),
                            "elems_per_s": w * (d << r) / (float(np.median(ts[2:])) * 1e-3),
                            "phase_ms_max_over_devices": {"FFT + blinding (peer loads)": ph[1], "leaf hashing": ph[3], "node levels": ph[4]}}
    ts, ph = run(dp, _ffi.PCS_DEVICE_PTRS | _ffi.PCS_MULTI_CE_GATHER, 2 + a.steps)
    res["device_inputs_ce_gather"] = {"ms": float(np.median(ts[2:])), "ms_min": float(min(ts[2:])), "cap_equal": bool(np.array_equal(cap, cap_expected)),
                                       "phase_ms_max_over_devices": {"FFT + blinding (incl. waits for the gather)": ph[1], "leaf hashing": ph[3], "node levels": ph[4]}}
    ts, ph = run(hp, _ffi.PCS_MULTI_CE_GATHER, 2 + a.steps)
    res["host_inputs_ce_gather"] = {"ms": float(np.median(ts[2:])), "ms_min": float(min(ts[2:])), "cap_equal": bool(np.array_equal(cap, cap_expected))}
    res["note"] = ("one process, one worker thread per GPU inside libpcs.so, no collective library; exchange = the first NTT pass reads the other "
                   "GPUs' coefficient blocks over NVLink in place (default), or -- *_ce_gather -- copy-engine gathers of polynomial group "
                   "c+1 under the LDE + hashing of group c; wall-clock of the synchronous C call incl. the cap D2H")
    del tens, full
    return res


def large_commit_bench(a, world, rank, dev, stream, lg_d=24):
    """BASELINE.json configs[4]: 135 polys x 2^24, rate_bits 3 (2^27 leaves, 145 GB of LDE rows) sharded over the box.
    The rows never leave the GPUs; parity at this size is sampled (SURVEY 8d): leaves fetched with their Merkle paths,
    (i) every path verified against the gathered cap by the CPU oracle, (ii) rows compared with a direct CPU evaluation
    of the polynomials at the leaf's domain point g * w_N^brev(leaf) (fri/verifier.rs:185-186 pins this order)."""
    import torch
    import torch.distributed as dist

    import oracle
    from helpers import P, brev, splitmix64_stream
    from plonky2_demo_b200.sharded import ShardedPolynomialBatch, ShardPlan

    w, r, cap_h = a.width, a.rate_bits, a.cap_height
    d = 1 << lg_d
    plan = ShardPlan(w, lg_d, r, cap_h, world, int(a.chunks) if str(a.chunks).isdigit() else a.chunks)
    mine = plan.local_polys(rank)
    t0 = time.perf_counter()
    host = np.empty((len(mine), d), dtype=np.uint64)
    for j, pj in enumerate(mine):
        host[j] = splitmix64_stream(0x5EED0000 + pj, d)
    local = torch.from_numpy(host.view(np.int64)).to(dev)
    gen_s = time.perf_counter() - t0
    times, batch = [], None
    for _ in range(3):
        if batch is not None:
            batch.free()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        batch = ShardedPolynomialBatch.from_coeffs(local, w, r, cap_h, partitioned=True, exchange=a.exchange, chunks=plan.sizes)
        e1.record(stream)
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
    n = plan.n_leaves
    rng = np.random.default_rng(7)
    leaves = sorted(set([0, n - 1] + [int(x) for x in rng.integers(0, n, size=3)]))
    rows = batch.get_rows(leaves)
    paths = batch.prove_many(leaves)
    ok_paths = True
    if rank == 0:
        for k, leaf in enumerate(leaves):
            ok_paths &= bool(oracle.merkle_verify(rows[k], leaf, batch.cap, paths[k].siblings))
    lg_n = lg_d + r
    wN = oracle.primitive_root_of_unity(lg_n)
    ok_rows, n_eval = True, min(2, len(mine))
    for k, leaf in enumerate(leaves):
        x = 7 * pow(wN, brev(leaf, lg_n), P) % P
        for j in range(n_eval):
            ok_rows &= int(rows[k][mine[j]]) == oracle.poly_eval(host[j], x)
    flag = torch.tensor([int(ok_rows)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res = {"workload": f"large commit: {w} polys x 2^{lg_d}, rate_bits {r}, cap_height {cap_h}, sharded over {world} GPUs",
           "ms": times, "best_ms": min(times), "elems_per_s": w * n / (min(times) * 1e-3), "lde_bytes": w * n * 8,
           "exchange": batch.exchange, "sampled_leaves": leaves, "merkle_paths_verify_against_cap": bool(ok_paths),
           "rows_equal_direct_cpu_evaluation": bool(flag.item()), "polys_evaluated_per_rank": n_eval,
           "input_generation_s": gen_s}
    batch.free()
    del local, host
    torch.cuda.empty_cache()
    return res


def run_ours(a):
    import torch
    import torch.distributed as dist

    import plonky2_demo_b200 as pcs
    from helpers import seeded_polys
    from plonky2_demo_b200 import _ffi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # A dedicated (non-default) stream shared by torch and the engine: the engine enqueues every kernel on
    # it, so torch.cuda.Event records on the same stream bracket exactly the engine's work.
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    pcs.init(local_rank, stream.cuda_stream)
    assert pcs.stream() == stream.cuda_stream
    L = _ffi.lib()

    w, lg_d, r, cap_h = a.width, a.lg_d, a.rate_bits, a.cap_height
    d, n = 1 << lg_d, 1 << (lg_d + r)
    elems = w * n

    # synthetic input: splitmix64(0x5EED0000 + j) stream per polynomial (SURVEY 8d).  world == 1: all W
    # polynomials; world > 1: this rank's block of the same W polynomials (plonky2_demo_b200/sharded.py)
    from plonky2_demo_b200.sharded import ShardedPolynomialBatch, ShardPlan

    def chunk_spec(x):
        return int(x) if str(x).isdigit() else x
    chunks = chunk_spec(a.chunks) if a.exchange not in ("peer", "alltoall") else 1
    plan = ShardPlan(w, lg_d, r, cap_h, world, chunks if world > 1 else 1)
    my_polys = plan.local_polys(rank) if world > 1 else list(range(w))
    w_loc = len(my_polys)
    host = torch.empty((w_loc, d), dtype=torch.int64, pin_memory=True)
    host_np = host.numpy().view(np.uint64)
    from helpers import splitmix64_stream
    for j, pj in enumerate(my_polys):
        host_np[j] = splitmix64_stream(0x5EED0000 + pj, d)
    dev_coeffs = host.to(dev, non_blocking=False)
    # end-to-end arm: its own chunking (and therefore its own block distribution of the same W polynomials)
    e2e_spec = a.e2e_chunks if a.e2e_chunks != "auto" else f"host:{0.75 if world >= 4 else 0.4}"
    e2e_chunks = chunk_spec(e2e_spec) if (a.exchange not in ("peer", "alltoall") and world > 1) else plan.sizes
    plan_e2e = ShardPlan(w, lg_d, r, cap_h, world, e2e_chunks if world > 1 else 1)
    if world > 1 and plan_e2e.sizes != plan.sizes and not a.no_e2e:
        polys_e2e = plan_e2e.local_polys(rank)
        host_e2e = torch.empty((len(polys_e2e), d), dtype=torch.int64, pin_memory=True)
        he = host_e2e.numpy().view(np.uint64)
        for j, pj in enumerate(polys_e2e):
            he[j] = splitmix64_stream(0x5EED0000 + pj, d)
    else:
        plan_e2e, host_e2e = plan, host
    cap_host = np.empty((1 << cap_h, 4), dtype=np.uint64)
    dev_ptrs = _ffi.dev_ptr_array(dev_coeffs.data_ptr(), w_loc, d)
    host_ptrs = _ffi.ptr_array([host_np[j] for j in range(w_loc)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class _Sharded:
        """adapter: free() like a raw handle"""
        def __init__(self, b):
            self.b = b

    def free(h):
        if isinstance(h, _Sharded):
            h.b.free()
        else:
            L.pcs_batch_free(h)

    def commit_device():
        if world > 1:
            return _Sharded(ShardedPolynomialBatch.from_coeffs(dev_coeffs, w, r, cap_h, partitioned=True, exchange=a.exchange,
                                                               chunks=plan.sizes))
        h = C.c_void_p()
        _ffi.check(L.pcs_commit_from_coeffs(dev_ptrs, w, lg_d, r, cap_h, None, 0, _ffi.PCS_DEVICE_PTRS, None, C.byref(h)))
        return h

    def commit_host():
        if world > 1:
            # streaming exchange: the pinned host block goes in as it is, chunk c+1 crosses PCIe / NVLink under the LDE of chunk c
            src = host_e2e if plan_e2e.chunks > 1 else host_e2e.to(dev, non_blocking=True)
            b = ShardedPolynomialBatch.from_coeffs(src, w, r, cap_h, partitioned=True, exchange=a.exchange, chunks=plan_e2e.sizes)
            cap_host[:] = b.cap
            return _Sharded(b)
        h = C.c_void_p()
        _ffi.check(L.pcs_commit_from_coeffs(host_ptrs, w, lg_d, r, cap_h, None, 0, 0, _ffi.ptr(cap_host), C.byref(h)))
        return h

    # ---- warm-up (also builds twiddle tables, fills the memory pool) ----
    for _ in range(max(a.warmup, 3)):
        free(commit_device())
    barrier()

    # ---- timed: K device-resident commits ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    _ffi.check(L.pcs_timing_totals(None, None, 1))  # reset the engine's per-phase event totals
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    e0.record(stream)
    prev = None
    for _ in range(a.steps):
        if prev is not None:
            free(prev)               # stream-ordered free: the next commit reuses this HBM
        prev = commit_device()       # world == 1: asynchronous (enqueues LDE passes, leaf hashing, node levels)
    e1.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    clocks = sampler.stop(t_wall0, t_wall1)
    ms_total = e0.elapsed_time(e1)
    cap_dev = np.empty((1 << cap_h, 4), dtype=np.uint64)
    prev_exchange = prev.b.exchange if world > 1 else "none"
    if world > 1:
        cap_dev[:] = prev.b.cap
    else:
        _ffi.check(L.pcs_batch_cap(prev, _ffi.ptr(cap_dev)))
    dump = None
    if a.dump_outputs:
        # read back while the last batch is alive; the reads launch no commit, so the phase totals below stay the timed ones
        depth = lg_d + r - cap_h
        idx = dump_sample(n, w, depth)
        if world > 1:
            rows = prev.b.get_rows(idx)
            paths = np.stack([p.siblings for p in prev.b.prove_many(idx)])
        else:
            rows = np.empty((idx.size, w), dtype=np.uint64)
            _ffi.check(L.pcs_batch_get_rows(prev, _ffi.ptr(idx), idx.size, _ffi.ptr(rows)))
            paths = np.empty((idx.size, depth, 4), dtype=np.uint64)
            _ffi.check(L.pcs_batch_prove_many(prev, _ffi.ptr(idx), idx.size, _ffi.ptr(paths)))
        dump = (idx, {"cap": cap_dev.copy(), "leaves": rows, "merkle_paths": paths})
    free(prev)
    ms5 = (C.c_float * 5)()
    ncommit = C.c_uint()
    _ffi.check(L.pcs_timing_totals(ms5, C.byref(ncommit), 1))
    assert ncommit.value == a.steps, (ncommit.value, a.steps)
    phase = np.array(list(ms5)) / a.steps
    if dump is not None and rank == 0:
        write_outputs(a.dump_outputs, *dump)

    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / a.steps
    value = elems * a.steps / (ms_total * 1e-3)   # one commitment of W*N elements per step, whatever the GPU count

    # ---- BASELINE configs[2]: the batched coset LDE alone, device resident (single GPU) ----
    lde_alone = None
    if world == 1:
        lde_out = torch.empty((w, n), dtype=torch.int64, device=dev)
        for _ in range(3):
            _ffi.check(L.pcs_coset_lde_dev(dev_ptrs, w, lg_d, r, 7, C.c_void_p(lde_out.data_ptr())))
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        g0.record(stream)
        for _ in range(a.steps):
            _ffi.check(L.pcs_coset_lde_dev(dev_ptrs, w, lg_d, r, 7, C.c_void_p(lde_out.data_ptr())))
        g1.record(stream)
        torch.cuda.synchronize()
        lde_alone = g0.elapsed_time(g1) / a.steps
        del lde_out

    # ---- PolynomialBatch::from_values at the same size (oracle.rs:43-65: IFFT of every column first), device resident ----
    from_values = None
    if world == 1 and not a.no_from_values:
        def commit_values():
            h = C.c_void_p()
            _ffi.check(L.pcs_commit_from_values(dev_ptrs, w, lg_d, r, cap_h, None, 0, _ffi.PCS_DEVICE_PTRS, None, None, C.byref(h)))
            return h
        for _ in range(2):
            free(commit_values())
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        _ffi.check(L.pcs_timing_totals(None, None, 1))
        v0.record(stream)
        for _ in range(a.steps):
            free(commit_values())
        v1.record(stream)
        torch.cuda.synchronize()
        fv_ms = v0.elapsed_time(v1) / a.steps
        fv5 = (C.c_float * 5)()
        _ffi.check(L.pcs_timing_totals(fv5, None, 1))
        from_values = {"workload": workload_name(a).replace("from_coeffs", "from_values"), "ms": fv_ms,
                       "elems_per_s": elems / (fv_ms * 1e-3), "ifft_ms": float(fv5[0]) / a.steps,
                       "note": "the seeded arrays taken as point VALUES; IFFT (size-d inverse NTT of every column) + the from_coeffs path"}

    # ---- SURVEY 8f N2/N3: the opening proof over the committed batch (single GPU) ----
    fri = None
    if world == 1 and not a.no_fri:
        fri = fri_opening_bench(pcs, w, lg_d, r, cap_h, dev_ptrs, a.steps, float(measured_peaks()[0]["hbm_gbs"]))

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region ----
    e2e = None
    if not a.no_e2e:
        for _ in range(2):
            free(commit_host())
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        tw0 = time.perf_counter()
        for _ in range(a.steps):
            h = commit_host()   # synchronous: returns once the cap is on the host
            free(h)
        f1.record(stream)
        barrier()
        tw1 = time.perf_counter()
        e2e_ms = max(f0.elapsed_time(f1), 1e3 * (tw1 - tw0))
        te = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_ms = float(te.item())
        assert np.array_equal(cap_host, cap_dev), "host-path and device-path caps differ"
        e2e = {"value": elems * a.steps / (e2e_ms * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(host_e2e.shape[0]) * d * 8, "d2h_bytes_per_step": (1 << cap_h) * 32,
               "exchange_chunks": plan_e2e.sizes if world > 1 else None,
               "ms_per_step": e2e_ms / a.steps,
               "note": "pinned host coefficients -> pcs_commit_from_coeffs (host pointers) -> Merkle cap on host; "
                       "LDE rows and digests stay device-resident behind the batch handle"}

    # ---- roofline of the dominant kernel (leaf hashing) + per-phase table ----
    peaks, peak_src = measured_peaks()
    peak = float(peaks["hbm_gbs"])
    wt = w
    n_loc = n // world                                       # leaves hashed by one rank's launches
    cap_loc = plan.local_cap_len() if world > 1 else (1 << cap_h)
    leaf_bytes = wt * n_loc * 8 + n_loc * 32                 # read every LDE element once, write one digest per leaf
    lde_bytes = w * d * 8 + w * n_loc * 8                    # read coefficients, write LDE (SURVEY 8d)
    node_bytes = 3 * 32 * (n_loc - cap_loc)                  # each node: read 2 children, write 1 digest
    commit_bytes = w * d * 8 + w * n * 8 + 2 * (n - (1 << cap_h)) * 32 + (1 << cap_h) * 32   # whole job (SURVEY 8d)
    leaf_ms, lde_ms, node_ms = phase[3], phase[1], phase[4]
    n_perm_leaf = n_loc * ((wt + 7) // 8) if wt > 4 else 0
    n_perm_node = n_loc - cap_loc
    roofline = {"bound": "hbm", "kernel": "k_hash_cols (Poseidon leaf hashing, 17 permutations per 135-element leaf)",
                "achieved": leaf_bytes / (leaf_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": leaf_bytes / (leaf_ms * 1e-3) / 1e9 / peak,
                "traffic": ncu_traffic(w, lg_d, r, world)[0], "traffic_source": ncu_traffic(w, lg_d, r, world)[1], "peak_source": peak_src,
                "algorithmic_bytes_per_launch": leaf_bytes, "launch_ms": leaf_ms,
                "note": "integer-pipe bound, not HBM bound: see int_pipe"}
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    int_pipe = {"permutations_per_s": (n_perm_leaf) / (leaf_ms * 1e-3),
                "clk_per_permutation_per_sm_lane": (leaf_ms * 1e-3) * sm_mhz * 1e6 * 148 / max(n_perm_leaf, 1),
                "sm_mhz_used": sm_mhz}
    # issue-slot view of the same launch: instructions per permutation are a property of the compiled kernel (ncu
    # smsp__inst_executed x 32 / permutations of the shipped k_hash_cols, profiles/r02_leafhash.md); an SM issues 4 x 32 thread-instructions per clock
    INSTR_PER_PERMUTATION, instr_src = leafhash_instr()
    issue_peak = 148 * 128 * sm_mhz * 1e6
    int_pipe.update({
        "thread_instr_per_permutation": INSTR_PER_PERMUTATION, "thread_instr_source": instr_src,
        "thread_instr_per_s": INSTR_PER_PERMUTATION * int_pipe["permutations_per_s"],
        "issue_peak_thread_instr_per_s": issue_peak,
        "issue_frac": INSTR_PER_PERMUTATION * int_pipe["permutations_per_s"] / issue_peak,
        "note": "the kernel's real ceiling: 64-bit modular arithmetic on 32-bit integer / FP64 pipes; measured pipe shares in "
                "profiles/r01_poseidon_v3.md and profiles/r02_forms.md (FP64 50 % + the IMAD family on one shared issue pipe, ALU 36 %)"})
    kernels = {
        "lde_standalone": None if lde_alone is None else {
            "workload": f"standalone batched coset LDE: {w} polys x 2^{lg_d}, rate_bits {r} (pcs_coset_lde_dev, 2 launches)",
            "ms": lde_alone, "elems_per_s": w * n / (lde_alone * 1e-3), "algorithmic_bytes": lde_bytes,
            "GBps": lde_bytes / (lde_alone * 1e-3) / 1e9, "frac_hbm": lde_bytes / (lde_alone * 1e-3) / 1e9 / peak,
            "note": "ALU-pipe bound (64-bit modular butterflies), see profiles/r01_ntt_v3.md"},
        "lde": {"ms": lde_ms, "algorithmic_bytes": lde_bytes, "GBps": lde_bytes / (lde_ms * 1e-3) / 1e9, "frac_hbm": lde_bytes / (lde_ms * 1e-3) / 1e9 / peak},
        "leaf_hash": {"ms": leaf_ms, "algorithmic_bytes": leaf_bytes, "GBps": roofline["achieved"], "frac_hbm": roofline["frac"], "permutations": n_perm_leaf},
        "node_levels": {"ms": node_ms, "algorithmic_bytes": node_bytes, "GBps": node_bytes / (node_ms * 1e-3) / 1e9, "permutations": n_perm_node},
        "fri_opening": fri,
        "commit": {"ms": ms_per_step, "algorithmic_bytes": commit_bytes, "GBps": commit_bytes / (ms_per_step * 1e-3) / 1e9,
                   "frac_hbm": commit_bytes / (ms_per_step * 1e-3) / 1e9 / peak},
    }

    lg_passes = (lg_d + 9) // 10 if lg_d else 1
    # per rank and commit: LDE passes (once per polynomial group of the streaming exchange) + leaf hashing + node levels
    lde_groups = plan.chunks if world > 1 else 1
    local_levels = (lg_d + plan.lg_cosets - plan.local_cap_height) if world > 1 else (lg_d + r - cap_h)
    # node levels: one launch per level while a level has more than 256 nodes per cap subtree, then ONE launch for the top of
    # every subtree; leaf hashing: one launch, or one per polynomial group of the streaming exchange (streaming sponge)
    def count_node_launches(n_leaves, lg_sub):
        """mirror of node_levels_dev (csrc/api.cu): levels of > 8192 nodes (throughput form) or of <= 8192 nodes with more than 64
        nodes per cap subtree (latency form) are one launch each, the rest of every subtree is ONE launch"""
        k, level = 0, 1
        while level <= lg_sub:
            nodes, left = n_leaves >> level, lg_sub - level
            if (left <= 6) if nodes <= 8192 else (left <= 8):
                break
            k += 1
            level += 1
        return k + (1 if level <= lg_sub else 0)
    node_launches = count_node_launches(n // world, local_levels)
    launches_per_step = lg_passes * lde_groups + lde_groups + node_launches
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64 (Goldilocks field, integer)", "data": "synthetic",
        "config": dict(bench_config(a), l2_policy="inputs larger than L2 (1.13 GB coefficients, 9.06 GB LDE per step); no flush needed",
                       parallelism=(f"one commitment sharded over {world} GPUs by coset block (contiguous leaf ranges); coefficient exchange = "
                                    f"{prev_exchange}; per-rank LDE + hashing; NCCL all-gather of the cap") if world > 1 else "single GPU"),
        "input_coeff_elems_per_s": value / (1 << r),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * a.steps,
        "roofline": roofline, "int_pipe": int_pipe, "kernels": kernels,
        "phase_ms": {"IFFT": phase[0], "FFT + blinding": phase[1], "transpose LDEs": phase[2], "leaf hashing": phase[3], "node levels": phase[4]},
    }
    out["kernels"]["from_values"] = from_values

    # ---- parity of what was just timed (every N): the benchmark checks itself against the oracle and the 1-GPU engine ----
    import oracle
    from helpers import seeded_polys as sp
    parity = {}
    lg_s = min(a.cpu_sample_lg_d, lg_d)
    if world == 1:
        small = sp(w, 1 << lg_s, base_seed=0x5EED0000)
        if rank == 0:
            ref_small = oracle.commit_from_coeffs(small, r, cap_h)
            b = pcs.PolynomialBatch.from_coeffs(small, r, False, cap_h)
            parity["cap_equal_to_oracle_at_sample_size"] = bool(np.array_equal(b.merkle_tree.cap.hashes, ref_small["cap"]))
            b.free()
            b = pcs.PolynomialBatch.from_values(oracle.fft(small), r, False, cap_h)
            parity["from_values_cap_equal_to_oracle_at_sample_size"] = bool(np.array_equal(b.merkle_tree.cap.hashes, ref_small["cap"]))
            b.free()
    else:
        # (i) the SHARDED path (real NCCL exchange, streaming chunks) against the CPU oracle at the sample size
        plan_s = ShardPlan(w, lg_s, r, cap_h, world, plan.sizes)
        mine_s = plan_s.local_polys(rank)
        loc = np.stack([splitmix64_stream(0x5EED0000 + pj, 1 << lg_s) for pj in mine_s]) if mine_s else np.empty((0, 1 << lg_s), np.uint64)
        bs = ShardedPolynomialBatch.from_coeffs(torch.from_numpy(loc.view(np.int64)).to(dev), w, r, cap_h, partitioned=True,
                                                exchange=a.exchange, chunks=plan_s.sizes)
        cap_s = np.array(bs.cap)
        leaf_s = (1 << (lg_s + r)) - 5
        row_s = bs.get_rows([leaf_s])[0]
        path_s = bs.prove(leaf_s)
        bs.free()
        if rank == 0:
            ref_small = oracle.commit_from_coeffs(sp(w, 1 << lg_s, base_seed=0x5EED0000), r, cap_h)
            parity["sharded_cap_equal_to_oracle_at_sample_size"] = bool(np.array_equal(cap_s, ref_small["cap"]))
            parity["sharded_row_equal_to_oracle"] = bool(np.array_equal(row_s, ref_small["leaves"][leaf_s]))
            parity["sharded_path_verifies_against_cap"] = bool(oracle.merkle_verify(row_s, leaf_s, cap_s, path_s.siblings))
        # (ii) the timed commitment itself against the SAME commitment on one GPU (the unsharded engine on rank 0)
        if rank == 0:
            full = torch.empty((w, d), dtype=torch.int64, pin_memory=True)
            fn = full.numpy().view(np.uint64)
            for j in range(w):
                fn[j] = splitmix64_stream(0x5EED0000 + j, d)
            cap_one = np.empty((1 << cap_h, 4), dtype=np.uint64)
            h1 = C.c_void_p()
            _ffi.check(L.pcs_commit_from_coeffs(_ffi.ptr_array([fn[j] for j in range(w)]), w, lg_d, r, cap_h, None, 0, 0,
                                                _ffi.ptr(cap_one), C.byref(h1)))
            L.pcs_batch_free(h1)
            parity["cap_equal_to_single_gpu"] = bool(np.array_equal(cap_dev, cap_one))
            parity["e2e_cap_equal_to_single_gpu"] = bool(np.array_equal(cap_host, cap_one)) if e2e is not None else None
            del full, fn
        dist.barrier()
    parity["lg_d_sample"] = lg_s
    out["parity_check"] = parity

    # ---- the same commitment through pcs_multi_*: ONE host process (rank 0) driving all N GPUs through the C ABI, the way a
    #      Rust prover would (no torch.distributed, no NCCL: peer loads fused into the first NTT pass) ----
    if world > 1 and not a.no_multi_in_process:
        dist.barrier()
        torch.cuda.synchronize()
        # the other ranks wait on the rendezvous STORE (a host-side wait): an NCCL barrier would leave a spinning kernel on their
        # GPUs, and kernels of two processes time-slice a GPU
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                out["kernels"]["multi_in_process"] = multi_in_process_bench(a, world, cap_dev)
            finally:
                store.set("pcs_multi_in_process_done", "1")
        else:
            store.wait(["pcs_multi_in_process_done"])
        dist.barrier()

    # ---- BASELINE configs[4]: one 135 x 2^24 commitment over the whole box ----
    if world > 1 and (a.large_commit == "on" or (a.large_commit == "auto" and world == 8 and lg_d == 20 and w == 135)):
        out["large_commit"] = large_commit_bench(a, world, rank, dev, stream)

    if rank == 0:
        if not a.no_cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(a)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    # the driver reads ONE JSON line from stdout: keep library chatter (e.g. NCCL's version banner) off it
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real_stdout, "w")
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
