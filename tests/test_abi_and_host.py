"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/pcs.h declares,
the host-side logic mirrors the reference, and the product never touches the oracle."""
import ast
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    from plonky2_demo_b200 import build

    return build.build()


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "pcs.h")) as f:
        h = f.read()
    return sorted(set(re.findall(r"PCS_API[^;(]*?\b(pcs_[a-z0-9_]+)\s*\(", h)))


def test_header_symbols_exported(built_lib):
    syms = _declared_symbols()
    assert len(syms) >= 25
    L = ctypes.CDLL(built_lib)
    for s in syms:
        assert hasattr(L, s), f"libpcs.so does not export {s}"
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (pcs_[a-z0-9_]+)", out))
    assert exported == set(syms), exported ^ set(syms)


def test_python_binding_matches_header(built_lib):
    import plonky2_demo_b200 as p

    assert sorted(p.SIGNATURES) == _declared_symbols()
    assert isinstance(p.lib(), ctypes.CDLL)


def test_no_cpu_fallback_without_device(built_lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    import plonky2_demo_b200 as p

    with pytest.raises(p.PcsError, match="no CPU fallback"):
        p.init(0)
    with pytest.raises(p.PcsError):
        p.PoseidonHash.hash_or_noop_batch(np.zeros((2, 8), dtype=np.uint64))
    with pytest.raises(p.PcsError):
        p.PolynomialBatch.from_coeffs(np.zeros((2, 8), dtype=np.uint64), 3, False, 0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "plonky2_demo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py"):
                tree = ast.parse(open(path).read())
                for node in ast.walk(tree):
                    names = []
                    if isinstance(node, ast.Import):
                        names = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        names = [node.module or ""]
                    assert not any(n.split(".")[0] == "oracle" for n in names), path
            elif f.endswith((".cu", ".cuh", ".h")):
                src = open(path).read()
                assert "oracle/" not in src and "liboracle" not in src, path
    out = subprocess.run(["ldd", os.path.join(pkg, "libpcs.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_fri_params_standard_recursion_config():
    import plonky2_demo_b200 as p

    cfg = p.CircuitConfig.standard_recursion_config()
    assert (cfg.num_wires, cfg.num_routed_wires, cfg.fri_config.rate_bits, cfg.fri_config.cap_height) == (135, 80, 3, 4)
    assert (cfg.fri_config.proof_of_work_bits, cfg.fri_config.num_query_rounds) == (16, 28)
    # reduction_strategies.rs:39-50 ConstantArityBits(4, 5)
    assert cfg.fri_config.fri_params(15, False).reduction_arity_bits == [4, 4, 4]
    assert cfg.fri_config.fri_params(20, False).reduction_arity_bits == [4, 4, 4, 4]
    assert cfg.fri_config.fri_params(3, False).reduction_arity_bits == []
    fp = cfg.fri_config.fri_params(15, False)
    assert fp.lde_bits() == 18 and fp.lde_size() == 1 << 18 and fp.final_poly_bits() == 3 and fp.total_arities() == 12
    assert cfg.fri_config.num_cap_elements() == 16
    assert p.PoseidonGoldilocksConfig.Hasher is p.PoseidonHash and p.PoseidonGoldilocksConfig.D == 2
    assert p.FriReductionStrategy.Fixed([3, 2, 1]).reduction_arity_bits(10, 3, 4, 28) == [3, 2, 1]


def test_host_helpers(golden):
    import plonky2_demo_b200 as p

    assert p.reverse_index_bits(np.arange(256, dtype=np.uint64)).tolist() == golden["kats"]["reverse_index_bits_256"]
    assert p.reverse_bits(0b01011, 5) == 0b11010  # plonky2/src/util/mod.rs:50
    assert p.log2_strict(1 << 20) == 20
    with pytest.raises(ValueError, match="Not a power of two: 12"):
        p.log2_strict(12)
    c = p.PolynomialCoeffs(np.arange(4, dtype=np.uint64))
    assert c.lde(2).coeffs.tolist() == [0, 1, 2, 3] + [0] * 12
    with pytest.raises(ValueError):
        c.padded(2)
    assert p.GOLDILOCKS_ORDER == golden["kats"]["field"]["order"]


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (CPU arm of the driver's contract): one JSON line with the contract's keys."""
    import json
    import sys

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample-lg-d", "8"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in rec, k
    assert rec["impl"] == "reference" and rec["unit"] == "elems/s" and rec["value"] > 0
    assert rec["cpu_baseline"]["kind"] == "port" and rec["e2e"]["h2d_bytes_per_step"] == 0
    # other ranks of a torchrun launch print nothing
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample-lg-d", "8"], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_rust_sys_binding_is_generated_from_header(built_lib):
    """rust/pcs-sys/src/lib.rs is what tools/gen_rust_sys.py makes of include/pcs.h, and declares exactly the exported symbols."""
    import importlib.util
    import re

    spec = importlib.util.spec_from_file_location("gen_rust_sys", os.path.join(ROOT, "tools", "gen_rust_sys.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    with open(os.path.join(ROOT, "rust", "pcs-sys", "src", "lib.rs")) as f:
        committed = f.read()
    assert committed == gen.generate(), "run `python tools/gen_rust_sys.py` after changing include/pcs.h"
    rust_fns = set(re.findall(r"pub fn (pcs_\w+)\(", committed))
    import plonky2_demo_b200 as p

    assert rust_fns == set(p.SIGNATURES), rust_fns ^ set(p.SIGNATURES)
    # pointer constness survives the translation (spot checks against the header)
    assert "coeffs_out: *const *mut u64" in committed            # uint64_t* const* coeffs_out
    assert "polys: *const *const u64" in committed               # const uint64_t* const* polys
    assert "out: *mut *mut pcs_batch" in committed               # pcs_batch** out
    assert "pub fn pcs_last_error() -> *const c_char;" in committed


def test_plonk_opening_shape_matches_reference_layout():
    """PlonkOpeningShape mirrors CommonCircuitData's ranges and get_fri_instance (circuit_data.rs:431-481,586-595) for the
    m = 64 demo: 4 oracles of 84 / 135 / 20 / 16 polynomials, everything opened at zeta, the 2 Zs also at g * zeta."""
    from plonky2_demo_b200.fri_prover import PlonkOpeningShape, ext_mul, primitive_root_of_unity

    s = PlonkOpeningShape(degree_bits=15, num_constants=4, num_routed_wires=80, num_wires=135, num_challenges=2,
                          num_partial_products=9, quotient_degree_factor=8)
    assert s.oracle_widths() == [84, 135, 20, 16]
    assert (list(s.constants_range()), s.sigmas_range().start, s.sigmas_range().stop) == ([0, 1, 2, 3], 4, 84)
    assert list(s.zs_range()) == [0, 1] and (s.partial_products_range().start, s.partial_products_range().stop) == (2, 20)
    zeta = (11, 22)
    inst = s.get_fri_instance(zeta)
    assert [o.num_polys for o in inst.oracles] == [84, 135, 20, 16] and not any(o.blinding for o in inst.oracles)
    b0, b1 = inst.batches
    assert b0.point == zeta and len(b0.polynomials) == 255
    assert [(p.oracle_index, p.polynomial_index) for p in b0.polynomials[:3]] == [(0, 0), (0, 1), (0, 2)]
    assert (b0.polynomials[84].oracle_index, b0.polynomials[84].polynomial_index) == (1, 0)
    assert (b0.polynomials[-1].oracle_index, b0.polynomials[-1].polynomial_index) == (3, 15)
    g = primitive_root_of_unity(15)
    assert pow(g, 1 << 15, 0xFFFFFFFF00000001) == 1 and pow(g, 1 << 14, 0xFFFFFFFF00000001) != 1
    assert b1.point == ext_mul((g, 0), zeta)
    assert [(p.oracle_index, p.polynomial_index) for p in b1.polynomials] == [(2, 0), (2, 1)]


def test_streaming_kernels_use_tma_bulk_copies(built_lib):
    """The HBM-facing opening-proof kernels stage their input with the TMA unit: the compiled object must contain the bulk
    copy (UBLKCP) and mbarrier (SYNCS) SASS (B200_PROFILING.md: the mnemonics that prove TMA), for sm_100a."""
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "plonky2_demo_b200", "build", "fri.o")
    if not os.path.exists(cuobjdump) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the object file is not available")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for kernel in ("k_eval_ext_tma", "k_reduce_polys_base_tma"):
        body = sass[sass.index(kernel):]
        body = body[: body.index("Function :", 10)] if "Function :" in body[10:] else body
        assert "UBLKCP" in body, kernel
        assert "SYNCS" in body, kernel


def _loop_bodies(sass, kernel):
    """Instruction lists of the backward-branch loops of one kernel in a `cuobjdump -sass` listing."""
    ins, on = [], False
    for line in sass.split("\n"):
        m = re.search(r"Function : (\S+)", line)
        if m:
            on = kernel in m.group(1)
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,6})\*/\s+(.*?);", line) if on else None
        if m:
            ins.append((int(m.group(1), 16), re.sub(r"^@!?U?P\d+\s+", "", m.group(2).strip())))
    loops = []
    for ad, t in ins:
        m = re.search(r"BRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?(0x[0-9a-f]+)", t)
        if m and int(m.group(1), 16) < ad:
            loops.append([x for a, x in ins if int(m.group(1), 16) <= a <= ad])
    return loops


def test_leaf_hash_kernel_instruction_budget(built_lib):
    """The reductions of csrc/gl64.cuh are written for what ptxas makes of them (profiles/r02_forms.md): the compiled
    leaf-hash kernel must keep the instruction counts the measurements were taken with -- one full Poseidon round in ~1018
    SASS instructions (1255 with the round 1-2 reductions), a partial-round pair in ~568 (610), five IMAD.WIDE per modular
    multiplication, the FP64 MDS network intact, and no spills."""
    import shutil

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "plonky2_demo_b200", "build", "leaf_hash.o")
    if not os.path.exists(cuobjdump) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the object file is not available")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    loops = sorted((l for l in _loop_bodies(sass, "k_hash_colsE") if len(l) > 300), key=len)
    assert len(loops) >= 2
    pair, full = loops[0], loops[1]                      # the two innermost round loops; the outer loops contain them
    count = lambda body, pre: sum(1 for t in body if t.split()[0].startswith(pre))
    assert 500 <= len(pair) <= 585, len(pair)
    assert 950 <= len(full) <= 1050, len(full)
    assert count(full, "IMAD.WIDE") == 12 * 4 * 5        # 12 S-boxes x 4 multiplications x (4 product + 1 reduction)
    assert count(full, "D") >= 190 and count(pair, "D") >= 400      # DADD / DFMA: the MDS layers run on the FP64 pipe
    res = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    usage = res[res.index("k_hash_colsE"):]
    m = re.search(r"REG:(\d+) STACK:(\d+)", usage)
    assert m and int(m.group(2)) == 0 and int(m.group(1)) <= 96, m and m.group(0)


def test_c_abi_smoke_links_with_gcc_and_fails_loudly_without_a_gpu(tmp_path):
    """tests/c_abi_smoke.c is plain C: it must compile and link against libpcs.so with gcc (no nvcc, no Python), and on a
    box without a GPU the very first call fails with the engine's "no CPU fallback" message instead of computing anything."""
    import subprocess

    from test_gpu_multi import build_c_smoke

    exe = build_c_smoke(tmp_path)
    try:
        import torch

        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("GPU present: the gpu-marked test runs the binary")
    r = subprocess.run([exe, "1", "4"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2
    assert "no CPU fallback" in r.stderr


def test_rust_shim_patches_apply_to_the_reference(tmp_path):
    """rust/plonky2-gpu-shim/patches/*.patch must apply cleanly to the reference's files (checked where /root/reference exists,
    i.e. in the build container; the GPU box has no reference tree), and gpu.rs may only call symbols the generated pcs-sys
    binding declares."""
    import shutil

    shim = os.path.join(ROOT, "rust", "plonky2-gpu-shim")
    with open(os.path.join(shim, "src", "gpu.rs")) as f:
        gpu = f.read()
    with open(os.path.join(ROOT, "rust", "pcs-sys", "src", "lib.rs")) as f:
        sys_rs = f.read()
    used = set(re.findall(r"sys::(pcs_[a-z0-9_]+)\s*\(", gpu))
    declared = set(re.findall(r"pub fn (pcs_[a-z0-9_]+)\s*\(", sys_rs))
    assert used and used <= declared, used - declared
    assert set(re.findall(r"sys::(PCS_[A-Z_]+)", gpu)) <= set(re.findall(r"pub const (PCS_[A-Z_0-9]+)", sys_rs))
    ref = "/root/reference"
    if not os.path.isdir(os.path.join(ref, "plonky2", "src", "fri")):
        pytest.skip("no reference tree on this machine")
    patches = sorted(p for p in os.listdir(os.path.join(shim, "patches")) if p.endswith(".patch"))
    assert len(patches) == 6
    for p in patches:
        with open(os.path.join(shim, "patches", p)) as f:
            target = f.readline().split()[1][2:]          # "--- a/<path>"
        dst = tmp_path / target
        dst.parent.mkdir(parents=True, exist_ok=True)
        shutil.copy(os.path.join(ref, target), dst)
        r = subprocess.run(["patch", "-p1", "--forward", "-i", os.path.join(shim, "patches", p)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, (p, r.stdout, r.stderr)
        assert 'feature = "cuda"' in dst.read_text() or "cuda =" in dst.read_text()
