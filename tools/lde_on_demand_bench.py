"""Resident vs on-demand commitments (PCS_LDE_ON_DEMAND) on one GPU: time and peak HBM of the commit, the two row paths of
get_rows, an lde_natural window, prove_openings, and 135 x 2^24.  Writes profiles/r03_lde_on_demand.{json,md}.

    python tools/lde_on_demand_bench.py [--reps 5] [--out profiles/r03_lde_on_demand]

Peak HBM is the high-water mark of the device's default memory pool (CU_MEMPOOL_ATTR_USED_MEM_HIGH, reset before each
commit): the engine allocates everything from that pool.  The caller's input tensors (torch's allocator) are not in it.
The group width and the get_rows crossover are compile-time constants (csrc/common.cuh); the variants measured here are
api.cu rebuilt with -DPCS_LDE_GROUP / -DPCS_ROWS_EVAL_MAX and linked with the in-tree objects into build/variants/, each run
in a worker process of its own (PCS_LIB)."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SHAPE = (135, 20, 3, 4)
GROUPS = (8, 16, 32, 64)
ROW_COUNTS = (1, 28, 128, 512, 2048)


# ---- build variants --------------------------------------------------------------------------------------------------
def variant(tag, defs):
    from plonky2_demo_b200 import build as B

    B.build()
    out = os.path.join(ROOT, "build", "variants", "on_demand")
    os.makedirs(out, exist_ok=True)
    obj, lib = os.path.join(out, f"api_{tag}.o"), os.path.join(out, f"libpcs_{tag}.so")
    src = os.path.join(B.CSRC, "api.cu")
    if not os.path.exists(lib) or os.path.getmtime(lib) < max(os.path.getmtime(B.LIB), os.path.getmtime(src)):
        subprocess.run([B.NVCC] + B.FLAGS + [f"-D{k}={v}" for k, v in defs.items()] + ["-c", src, "-o", obj], check=True)
        objs = [os.path.join(B.BUILD, f) for f in sorted(os.listdir(B.BUILD)) if f.endswith(".o") and f != "api.o"]
        subprocess.run([B.NVCC, "-shared", "-ccbin", "/usr/bin/g++", "-o", lib, obj] + objs +
                       ["-lcudart_static", "-ldl", "-lrt", "-lpthread"], check=True)
    return lib


# ---- measurement helpers (worker side) -------------------------------------------------------------------------------
class Pool:
    """The default memory pool's used-memory high-water mark, through the driver API."""

    def __init__(self):
        self.cu = C.CDLL("libcuda.so.1")
        assert self.cu.cuInit(0) == 0
        dev = C.c_int()
        assert self.cu.cuDeviceGet(C.byref(dev), 0) == 0
        self.pool = C.c_void_p()
        assert self.cu.cuDeviceGetDefaultMemPool(C.byref(self.pool), dev) == 0

    def reset(self):
        z = C.c_uint64(0)
        assert self.cu.cuMemPoolSetAttribute(self.pool, 8, C.byref(z)) == 0   # CU_MEMPOOL_ATTR_USED_MEM_HIGH

    def high(self):
        v = C.c_uint64()
        assert self.cu.cuMemPoolGetAttribute(self.pool, 8, C.byref(v)) == 0
        return v.value


def stats(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def worker(what, reps):
    import numpy as np
    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    p.init(0)
    L, pool = _ffi.lib(), Pool()
    res = {}

    def commit(x, w, lg_d, r, cap_h, flags, host=None):
        h = C.c_void_p()
        d = 1 << lg_d
        ptrs = host if host is not None else _ffi.dev_ptr_array(x.data_ptr(), w, d)
        L.pcs_synchronize()
        pool.reset()
        t0 = time.perf_counter()
        _ffi.check(L.pcs_commit_from_coeffs(ptrs, w, lg_d, r, cap_h, None, 0, flags, None, C.byref(h)))
        _ffi.check(L.pcs_synchronize())
        return h, (time.perf_counter() - t0) * 1e3, pool.high()

    w, lg_d, r, cap_h = SHAPE
    d, n = 1 << lg_d, 1 << (lg_d + r)
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randint(0, 1 << 62, (w, d), dtype=torch.int64, device="cuda", generator=gen)
    dev, od = _ffi.PCS_DEVICE_PTRS, _ffi.PCS_LDE_ON_DEMAND
    if what == "commit":
        xh = x.cpu().pin_memory()
        host = (_ffi.u64p * w)(*[C.cast(C.c_void_p(xh.data_ptr() + 8 * j * d), _ffi.u64p) for j in range(w)])
        for src in ("device", "pinned"):
            for _ in range(2):   # warm-up
                for f in (0, od):
                    h, _, _ = commit(x, w, lg_d, r, cap_h, f | (dev if src == "device" else 0), None if src == "device" else host)
                    L.pcs_batch_free(h)
            t = {"resident": [], "on_demand": []}
            peak = {}
            for _ in range(reps):   # alternate the two modes
                for name, f in (("resident", 0), ("on_demand", od)):
                    h, ms, hi = commit(x, w, lg_d, r, cap_h, f | (dev if src == "device" else 0), None if src == "device" else host)
                    t[name].append(ms)
                    peak[name] = hi
                    L.pcs_batch_free(h)
            res[src] = {k: {"ms": stats(v), "peak_hbm_bytes": peak[k]} for k, v in t.items()}
    elif what == "group":
        for _ in range(2):
            h, _, _ = commit(x, w, lg_d, r, cap_h, dev | od)
            L.pcs_batch_free(h)
        ts, hi = [], 0
        for _ in range(reps):
            h, ms, hi = commit(x, w, lg_d, r, cap_h, dev | od)
            ts.append(ms)
            L.pcs_batch_free(h)
        res = {"ms": stats(ts), "peak_hbm_bytes": hi}
    elif what == "rows":
        hr, _, _ = commit(x, w, lg_d, r, cap_h, dev)
        ho, _, _ = commit(x, w, lg_d, r, cap_h, dev | od)
        rng = np.random.default_rng(7)
        for m in ROW_COUNTS:
            idx = np.ascontiguousarray(rng.integers(0, n, size=m).astype(np.uint64))
            out = {k: np.empty((m, w), dtype=np.uint64) for k in ("r", "o")}
            t = {"resident": [], "on_demand": []}
            for rep in range(reps + 1):
                for name, h, o in (("resident", hr, out["r"]), ("on_demand", ho, out["o"])):
                    t0 = time.perf_counter()
                    _ffi.check(L.pcs_batch_get_rows(h, _ffi.ptr(idx), m, _ffi.ptr(o)))
                    if rep:
                        t[name].append((time.perf_counter() - t0) * 1e3)
            assert np.array_equal(out["r"], out["o"])
            res[str(m)] = {k: stats(v) for k, v in t.items()}
        # a window of the quotient loop: 2^20 consecutive natural points, step 1
        cnt = 1 << 20
        out = {k: np.empty((cnt, w), dtype=np.uint64) for k in ("r", "o")}
        t = {"resident": [], "on_demand": []}
        for rep in range(3):
            for name, h, o in (("resident", hr, out["r"]), ("on_demand", ho, out["o"])):
                t0 = time.perf_counter()
                _ffi.check(L.pcs_batch_lde_natural(h, 0, 1, cnt, _ffi.ptr(o)))
                if rep:
                    t[name].append((time.perf_counter() - t0) * 1e3)
        assert np.array_equal(out["r"], out["o"])
        res["lde_natural_2^20_step1"] = {k: stats(v) for k, v in t.items()}
        L.pcs_batch_free(hr)
        L.pcs_batch_free(ho)
    elif what == "openings":
        from plonky2_demo_b200.fri_prover import (Challenger, FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo,
                                                  prove_openings)

        xn = x.cpu().numpy().view(np.uint64)
        inst = FriInstanceInfo([FriOracleInfo(w, False)], [FriBatchInfo((3, 5), [FriPolynomialInfo(0, j) for j in range(w)])])
        cfg = p.FriConfig(r, cap_h, 8, p.FriReductionStrategy.ConstantArityBits(4, 5), 28)
        params = cfg.fri_params(lg_d, False)
        t = {"resident": [], "on_demand": []}
        proofs = {}
        for rep in range(reps + 1):
            for name, on in (("resident", False), ("on_demand", True)):
                b = p.PolynomialBatch.from_coeffs(xn, r, False, cap_h, keep_coeffs=True, lde_on_demand=on)
                ch = Challenger()
                ch.observe_cap(b.merkle_tree.cap.hashes)
                _ffi.check(L.pcs_synchronize())
                t0 = time.perf_counter()
                proofs[name] = prove_openings(inst, [b], ch, params)
                if rep:
                    t[name].append((time.perf_counter() - t0) * 1e3)
                b.free()
        a, bq = proofs["resident"], proofs["on_demand"]
        assert all(np.array_equal(e1, e2) for r1, r2 in zip(a.query_round_proofs, bq.query_round_proofs)
                   for (e1, _), (e2, _) in zip(r1.initial_trees_proof.evals_proofs, r2.initial_trees_proof.evals_proofs))
        res = {k: stats(v) for k, v in t.items()}
    elif what == "large":
        del x
        torch.cuda.empty_cache()
        lg = 24
        xl = torch.randint(0, 1 << 62, (w, 1 << lg), dtype=torch.int64, device="cuda", generator=gen)
        ts, hi = [], 0
        for _ in range(2):
            h, ms, hi = commit(xl, w, lg, r, cap_h, dev | od)
            ts.append(ms)
            L.pcs_batch_free(h)
        res = {"ms": stats(ts[1:]), "first_ms": ts[0], "peak_hbm_bytes": hi}
    p.shutdown()
    print("RESULT " + json.dumps(res))


def run_worker(what, lib, reps):
    env = dict(os.environ, PCS_LIB=lib)
    r = subprocess.run([sys.executable, __file__, "--worker", what, "--reps", str(reps)], env=env, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f"worker {what} failed:\n{r.stdout}\n{r.stderr}")
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1][7:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lde_on_demand"))
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.reps)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    from plonky2_demo_b200 import build as B

    res = {"gpu": q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown", "shape": SHAPE, "reps": a.reps}
    res["group_width"] = {str(g): run_worker("group", variant(f"g{g}", {"PCS_LDE_GROUP": g}), a.reps) for g in GROUPS}
    res["commit"] = run_worker("commit", B.build(), a.reps)
    res["get_rows_eval"] = run_worker("rows", variant("eval", {"PCS_ROWS_EVAL_MAX": 1 << 30}), a.reps)
    res["get_rows_regen"] = run_worker("rows", variant("regen", {"PCS_ROWS_EVAL_MAX": 0}), a.reps)
    res["prove_openings"] = run_worker("openings", B.build(), min(a.reps, 3))
    res["large_135x2^24"] = run_worker("large", B.build(), 1)
    with open(a.out + ".json", "w") as f:
        json.dump(res, f, indent=1)
    gb = 1e9
    lines = [f"# Resident vs on-demand commitments ({res['gpu']})", "",
             f"Shape {SHAPE[0]} x 2^{SHAPE[1]}, rate {SHAPE[2]}, cap {SHAPE[3]}; medians of {a.reps} runs [min-max]; peak HBM = "
             "default pool high-water mark.", "", "| group width G | on-demand commit ms | peak HBM GB |", "|---|---|---|"]
    for g, v in res["group_width"].items():
        lines.append(f"| {g} | {v['ms']['median']:.2f} [{v['ms']['min']:.2f}-{v['ms']['max']:.2f}] | {v['peak_hbm_bytes'] / gb:.2f} |")
    lines += ["", "| input | mode | commit ms | peak HBM GB |", "|---|---|---|---|"]
    for src, v in res["commit"].items():
        for mode, m in v.items():
            lines.append(f"| {src} | {mode} | {m['ms']['median']:.2f} [{m['ms']['min']:.2f}-{m['ms']['max']:.2f}] | "
                         f"{m['peak_hbm_bytes'] / gb:.2f} |")
    lines += ["", "| rows | resident ms | evaluated ms | regenerated ms |", "|---|---|---|---|"]
    for m in ROW_COUNTS:
        e, g = res["get_rows_eval"][str(m)], res["get_rows_regen"][str(m)]
        lines.append(f"| {m} | {e['resident']['median']:.2f} | {e['on_demand']['median']:.2f} | {g['on_demand']['median']:.2f} |")
    ln = res["get_rows_eval"]["lde_natural_2^20_step1"]
    lines += ["", f"lde_natural, 2^20 points at step 1: resident {ln['resident']['median']:.1f} ms, "
              f"on demand {ln['on_demand']['median']:.1f} ms.",
              f"prove_openings (one oracle, 28 queries): resident {res['prove_openings']['resident']['median']:.1f} ms, "
              f"on demand {res['prove_openings']['on_demand']['median']:.1f} ms.",
              f"135 x 2^24 on demand: {res['large_135x2^24']['ms']['median']:.1f} ms, "
              f"peak HBM {res['large_135x2^24']['peak_hbm_bytes'] / gb:.1f} GB."]
    with open(a.out + ".md", "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
