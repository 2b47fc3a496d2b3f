"""A tiny interpreter for the PTX subset used by the inline-asm field arithmetic in csrc/gl64.cuh (integer add / sub with the
carry flag, 32x32 wide multiplies, shifts, 64-bit packs).  It lets the CPU test-suite check the ALGORITHM of every device
reduction against big-int arithmetic without a GPU (ptxas and the hardware are then
covered by the `-m gpu` field-grid and Poseidon KAT tests).  Test infrastructure only."""
import re
import subprocess

M32, M64 = (1 << 32) - 1, (1 << 64) - 1


def preprocess(path, defines):
    """Run the C preprocessor over a header (comments dropped, `defines` applied) so that only code is left to parse."""
    cmd = ["cpp", "-P", "-x", "c++", "-undef"] + [f"-D{k}={v}" for k, v in defines.items()] + [path]
    return subprocess.run(cmd, capture_output=True, text=True, check=True).stdout


def _in_string(src, start, pos):
    return src.count('"', start, pos) % 2 == 1


def extract_asm(src, func):
    """(asm text, [(constraint, c_expr) outputs], [(constraint, c_expr) inputs]) of the asm statement inside `func`."""
    m = re.search(r"\b" + re.escape(func) + r"\s*\([^)]*\)\s*\{", src)
    assert m, func
    depth, e = 1, m.end()
    while depth:                      # the function's own body only
        depth += {"{": 1, "}": -1}.get(src[e], 0) if not _in_string(src, m.end(), e) else 0
        e += 1
    body = src[m.end():e]
    if "asm(" not in body:
        return None
    a = body.index("asm(")
    depth, i = 0, a + 3
    while True:
        if body[i] == "(":
            depth += 1
        elif body[i] == ")":
            depth -= 1
            if depth == 0:
                break
        i += 1
    stmt = body[a + 4:i]
    # split the string literal part from the operand lists at the first ':' outside quotes
    parts, cur, inq = [], "", False
    k = 0
    while k < len(stmt):
        ch = stmt[k]
        if ch == '"' and (k == 0 or stmt[k - 1] != "\\"):
            inq = not inq
        if ch == ":" and not inq:
            parts.append(cur)
            cur = ""
        else:
            cur += ch
        k += 1
    parts.append(cur)
    text = "".join(re.findall(r'"((?:[^"\\]|\\.)*)"', parts[0]))
    text = text.replace("\\n", "\n").replace("\\t", " ")
    ops = lambda s: [(c, e.strip()) for c, e in re.findall(r'"([^"]+)"\s*\(((?:[^()]|\([^()]*\))*)\)', s)]
    return text, ops(parts[1]) if len(parts) > 1 else [], ops(parts[2]) if len(parts) > 2 else []


def _compile(text):
    """Parse an asm block once: a list of (kind, dst, srcs, bits, flags) tuples the interpreter loop can run quickly."""
    prog, regs = [], []
    for line in text.split(";"):
        line = re.sub(r"//.*", "", line).strip()
        while line.startswith("{") and not line.startswith("{%"):
            line = line[1:].strip()
        line = line.rstrip("}").strip() if not re.search(r"\{[^}]*\}\s*$", line) else line
        if not line or line == "}":
            continue
        if line.startswith(".reg"):
            regs += [n.strip() for n in line.split(None, 2)[2].split(",")]
            continue
        op, rest = line.split(None, 1)
        if op == "mov.b64":
            dst, src = [x.strip() for x in re.split(r",(?![^{]*\})", rest, 1)]
            if dst.startswith("{"):
                lo, hi = [x.strip() for x in dst.strip("{}").split(",")]
                prog.append(("unpack", (lo, hi), (src,), 64, 0))
            else:
                lo, hi = [x.strip() for x in src.strip("{}").split(",")]
                prog.append(("pack", dst, (lo, hi), 64, 0))
            continue
        a = [x.strip() for x in rest.split(",")]
        srcs = tuple(int(x, 0) if re.fullmatch(r"-?(0x[0-9a-fA-F]+|\d+)", x) else x for x in a[1:])
        bits = 64 if op.endswith("64") and not op.startswith(("mul.wide", "cvt")) else 32
        base = op.split(".")[0]
        cc = ".cc" in op
        if base in ("add", "addc", "sub", "subc"):
            prog.append((base, a[0], srcs, bits, cc))
        elif base in ("mad", "madc"):
            prog.append((base, a[0], srcs, 32, (cc, ".hi" in op)))
        elif op == "mul.wide.u32":
            prog.append(("mulwide", a[0], srcs, 64, 0))
        elif op == "cvt.u64.u32":
            prog.append(("cvt", a[0], srcs, 64, 0))
        elif op == "neg.s32":
            prog.append(("neg", a[0], srcs, 32, 0))
        elif op == "shr.s32":
            prog.append(("sar", a[0], srcs, 32, 0))
        else:
            raise NotImplementedError(op)
    return prog, regs


_CACHE = {}


def _exec(text, r):
    if text not in _CACHE:
        _CACHE[text] = _compile(text)
    prog, regs = _CACHE[text]
    for n in regs:
        r[n] = 0
    cf = 0
    for kind, d, s, bits, fl in prog:
        v = [x if isinstance(x, int) else r[x] for x in s]
        mask = (1 << bits) - 1
        if kind == "add" or kind == "addc":
            t = (v[0] & mask) + (v[1] & mask) + (cf if kind == "addc" else 0)
            r[d] = t & mask
            if fl:
                cf = t >> bits
        elif kind == "sub" or kind == "subc":
            t = (v[0] & mask) - (v[1] & mask) - (cf if kind == "subc" else 0)
            r[d] = t & mask
            if fl:
                cf = 1 if t < 0 else 0
        elif kind == "mad" or kind == "madc":
            p = (v[0] & M32) * (v[1] & M32)
            t = ((p >> 32) if fl[1] else (p & M32)) + (v[2] & M32) + (cf if kind == "madc" else 0)
            r[d] = t & M32
            if fl[0]:
                cf = t >> 32
        elif kind == "mulwide":
            r[d] = (v[0] & M32) * (v[1] & M32)
        elif kind == "cvt":
            r[d] = v[0] & M32
        elif kind == "neg":
            r[d] = (-v[0]) & M32
        elif kind == "sar":
            x = v[0] & M32
            x = x - (1 << 32) if x >> 31 else x
            r[d] = (x >> v[1]) & M32
        elif kind == "unpack":
            r[d[0]], r[d[1]] = v[0] & M32, (v[0] >> 32) & M32
        elif kind == "pack":
            r[d] = (v[0] & M32) | ((v[1] & M32) << 32)
    return r


def run_asm(text, outs, ins, env):
    """Evaluate one asm statement; env maps C expressions (as written in the operand lists) to integers.  Returns env updated
    with the output expressions.  Carry flag semantics as in the PTX ISA: add.cc / addc carry, sub.cc / subc borrow."""
    r = {}
    for k, (c, e) in enumerate(outs + ins):
        r[f"%{k}"] = env.get(e, 0) if (c.startswith("+") or not c.startswith("=")) else 0
    _exec(text, r)
    res = dict(env)
    for k, (c, e) in enumerate(outs):
        res[e] = r[f"%{k}"]
    return res
