"""The device field primitives at their carry and wrap boundaries, against exact integer arithmetic.

tests/field_probe.cu runs single primitives of the Goldilocks fast path (gl.cuh, GlField in field_policy.cuh) and the BN254
carry chains (bn254.cuh) on case tables built here. Random operands almost never take the rare corrections (the borrow of
acc_reduce, the final canonicalisation, a carry out of gl_add_cs, t == r in fr_cond_sub_dev), so the tables are built from
boundary values and from accumulator states solved to land on 0, p - 1 and p; test_case_tables_take_every_branch checks, on
the CPU, that every branch is taken. Each table stays inside the contract its primitive states in gl.cuh / bn254.cuh
(which inputs may be lazy, the accumulator capacity, the bound on e4) and reaches that contract's limit."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hyper-greco_b200", "csrc")
PROBE_SRC = os.path.join(ROOT, "tests", "field_probe.cu")

P = 2**64 - 2**32 + 1
EPS = 2**32 - 1
M64 = 2**64 - 1
M32 = 2**32 - 1
E4_MAX = 2**32 - 3   # acc_reduce is exact for e4 <= E4_MAX (gl.cuh)
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
BN_RM = 2**256 % BN_R                 # R mod r: the Montgomery form of 1
BN_RINV = pow(2**256, -1, BN_R)

# op codes and row widths of field_probe.cu
OP_ACC_REDUCE, OP_ACC_RUN, OP_XACC, OP_SUB_ADD, OP_MUL, OP_FOLD, OP_LINE, OP_CHAIN, OP_FR, OP_FR_COND_SUB, OP_FR_CANON = range(11)
IN_WORDS = [5, 9, 20, 2, 4, 10, 7, 8, 8, 5, 4]
OUT_WORDS = [1, 1, 2, 3, 7, 6, 7, 8, 16, 4, 8]

GL_LAZY = [0, 1, 2, EPS - 1, EPS, 2**32, 2**32 + 1, 2**63 - 1, 2**63, P - 2, P - 1, P, P + 1, M64 - 1, M64]
GL_CANON = [v for v in GL_LAZY if v < P]


# ------------------------------------------------------------------------------------------------ exact references
def acc_value(s):
    e01, e23, o01, e4, o2 = s
    return e01 + (e23 << 64) + (e4 << 128) + ((o01 + (o2 << 64)) << 32)


def ext_mul(a, b):
    return ((a[0] * b[0] + 7 * a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def fr_limbs(v, n=4):
    return [(v >> (64 * j)) & M64 for j in range(n)]


def fr_int(row):
    return sum(int(x) << (64 * j) for j, x in enumerate(row))


# ------------------------------------------------------------------------------------------------ branch conditions, transliterated from the device code
def acc_reduce_branches(s):
    """(borrow in gl_sub_cs(lo, s1), carry of t0 + t1, final gl_canon subtract, merged top word c) of acc_reduce (gl.cuh)."""
    e01, e23, o01, e4, o2 = s
    v = (e01 >> 32) + ((e23 & M64) << 32) + (e4 << 96) + o01 + (o2 << 64)   # e1 e2 e3 c after the odd-column merge
    e1, e2, e3, c = v & M32, (v >> 32) & M32, (v >> 64) & M32, v >> 96
    lo, s1 = (e01 & M32) | (e1 << 32), e3 | (c << 32)
    borrow = lo < s1
    t0 = (lo - s1 - (EPS if borrow else 0)) & M64
    t1 = (e2 << 32) - e2
    carry = t0 + t1 > M64
    r = (t0 + t1 + (EPS if carry else 0)) & M64
    return borrow, carry, r >= P, c


def sub_cs(a, b):
    return (a - b - (EPS if a < b else 0)) & M64


def add_cs(a, b):
    return (a + b + (EPS if a + b > M64 else 0)) & M64


# ------------------------------------------------------------------------------------------------ case tables
def _lazy(rng):
    return rng.choice(GL_LAZY) if rng.random() < 0.7 else rng.getrandbits(64)


def _canon(rng):
    return rng.choice(GL_CANON) if rng.random() < 0.6 else rng.randrange(P)


def _state(rng, k=0):
    """An accumulator state with room for k more acc_mad calls before acc_reduce: e4 <= E4_MAX - k, o2 <= 2^32 - 1 - 2k."""
    e4_top, o2_top = E4_MAX - k, M32 - 2 * k
    e4 = rng.choice([0, 1, 2**31 - 1, 2**31, e4_top, rng.randrange(e4_top + 1), rng.getrandbits(3)])
    o2 = rng.choice([0, 1, o2_top, rng.randrange(o2_top + 1), rng.getrandbits(3)])
    return [_lazy(rng), _lazy(rng), _lazy(rng), e4, o2]


def cases_acc_reduce():
    rng = random.Random(1)
    rows = [_state(rng) for _ in range(3000)]
    # solved states: o = 0, so lo = e01 and s1 = e3 + 2^32 e4; pick e01 so that the value is 0, 1 or p - 1, once as the
    # smallest representative (borrow when below s1) and once p higher (no borrow, or the final subtract of gl_canon)
    for _ in range(200):
        e23, e4 = _lazy(rng), rng.choice([0, 1, 2**31, E4_MAX, rng.randrange(E4_MAX + 1)])
        s1, t1 = (e23 >> 32) | (e4 << 32), ((e23 & M32) << 32) - (e23 & M32)
        for target in (0, 1, P - 1):
            lo = (target + s1 - t1) % P
            rows.append([lo, e23, 0, e4, 0])
            if lo + P <= M64:
                rows.append([lo + P, e23, 0, e4, 0])
    # the largest representatives: e4 = E4_MAX with every lower word all ones (the merge carries into c: c = 2^32 - 2)
    for e01 in (0, 1, P - 1, P, M64):
        rows.append([e01, M64, M64, E4_MAX, M32])
        rows.append([e01, M64, M64, E4_MAX - 1, M32])
    for v in (0, 1, P - 2, P - 1, P, P + 1, M64):
        rows.append([v, 0, 0, 0, 0])
    return rows


def _run_limit_row(e01, e23, o01, x, y, z, reps):
    """An acc_mad / acc_add run that ends exactly at the capacity limits: o2 = 2^32 - 1 and e4 = E4_MAX."""
    cross = (x & M32) * (y >> 32) + (x >> 32) * (y & M32)
    even = (x & M32) * (y & M32) + ((x >> 32) * (y >> 32) << 64) + z
    o2 = M32 - ((o01 + reps * cross) >> 64)
    e_lo = e01 + (e23 << 64) + reps * even                # e4 grows by e_lo >> 128
    e4 = E4_MAX - (e_lo >> 128)
    return [e01, e23, o01, e4, o2, x, y, z, reps]


def cases_acc_run():
    rng = random.Random(2)
    rows = []
    for reps in (1, 2, 255, 1 << 16, (1 << 24) - 1):
        rows.append([0, 0, 0, 0, 0, M64, M64, M64, reps])                 # from zero, the largest operands
        rows.append(_run_limit_row(M64, M64, M64, M64, M64, M64, reps))
        rows.append(_run_limit_row(0, 0, 0, M64, M64, 0, reps))
        rows.append(_run_limit_row(P, P - 1, 0, P - 1, P, P, reps))
    for _ in range(200):
        reps = rng.choice([1, 2, 3, 17, 1000])
        x, y, z = _lazy(rng), _lazy(rng), _lazy(rng)
        rows.append(_run_limit_row(_lazy(rng), _lazy(rng), _lazy(rng), x, y, z, reps) if rng.random() < 0.5
                    else _state(rng, 2 * reps) + [x, y, z, reps])
    return rows


def cases_xacc():
    rng = random.Random(3)
    rows = []
    for i in range(1500):
        # a00 takes x0 y0, x0 yb and 7 * reduce(a11); a11 takes x1 y1; ax takes x0 y1, x1 y0, x1 yb
        a00, a11, ax = _state(rng, 3), _state(rng, 1), _state(rng, 3)
        if i < 16:
            a00, a11, ax = [M64, M64, M64, E4_MAX - 3, M32 - 6], [M64, M64, M64, E4_MAX - 1, M32 - 2], [M64, M64, M64, E4_MAX - 3, M32 - 6]
        rows.append(a00 + a11 + ax + [_lazy(rng) for _ in range(5)])
    return rows


def cases_sub_add():
    rng = random.Random(4)
    rows = [[a, b] for a in GL_LAZY for b in GL_CANON]
    rows += [[_lazy(rng), _canon(rng)] for _ in range(2000)]
    return rows


def cases_mul():
    rng = random.Random(5)
    rows = [[a, b, c, d] for a in GL_LAZY for c in GL_LAZY for b, d in ((a, c), (M64, P - 1), (0, 1))]
    rows += [[_lazy(rng) for _ in range(4)] for _ in range(1000)]
    rows += [[_canon(rng) for _ in range(4)] for _ in range(1000)]
    return rows


def cases_fold():
    rng = random.Random(6)
    rows = []
    for i in range(3000):
        a0, a1, r, c = [_canon(rng), _canon(rng)], [_canon(rng), _canon(rng)], [_canon(rng), _canon(rng)], [_canon(rng), _canon(rng)]
        cr = list(ext_mul(c, r)) if i % 2 == 0 else [_canon(rng), _canon(rng)]
        rows.append(a0 + a1 + r + c + cr)
    ends = [0, 1, P - 1]
    for a, b, r in ((a, b, r) for a in ends for b in ends for r in ends):
        rows.append([a, a, b, b, r, r, r, r] + list(ext_mul([r, r], [r, r])))
    return rows


def cases_line():
    rng = random.Random(7)
    rows = [[lo, lo, hi, hi, lo, hi, q] for lo in GL_CANON for hi in GL_CANON for q in (0, P - 1)]
    rows += [[_canon(rng) for _ in range(7)] for _ in range(2000)]
    return rows


def cases_chain():
    rng = random.Random(8)
    # (lo, hi) = (p - 1, p - 2) makes at_m1 = p, a non-canonical zero; (0, p - 1) and (p - 1, 0) take the borrow of slope / at_m1
    pairs = [(P - 1, P - 2), (0, P - 1), (P - 1, 0), (1, P - 1), (P - 1, P - 1), (0, 0), (P - 2, P - 1)]
    rows = []
    for t in pairs:
        for l in pairs:
            for r in pairs:
                rows.append(list(t) + list(l) + list(r) + [rng.choice(GL_CANON), rng.choice(GL_CANON)])
    rows += [[_canon(rng) for _ in range(8)] for _ in range(2000)]
    return rows


def _fr_pool():
    r = BN_R
    pool = [0, 1, 2, r - 1, r - 2, (r - 1) // 2, (r + 1) // 2, BN_RM, r - BN_RM, (2 * BN_RM) % r]
    pool += [M64 << (64 * j) for j in range(3)]                    # 2^64 - 1 in one limb below r's top limb
    pool += [(2**192 - 1) | ((r >> 192) - 1) << 192]              # all ones below a top limb of FR_MOD3 - 1
    for j in range(3):                                            # top limb = FR_MOD3, lower limbs at and around r's
        pool += [r - (1 << (64 * j)), r - (2 << (64 * j)), r - 1 - (1 << (64 * j))]
    pool += [(r >> 192) << 192, ((r >> 192) << 192) | M64]
    return sorted(set(v for v in pool if 0 <= v < r))


def cases_fr():
    rng = random.Random(9)
    pool = _fr_pool()
    rows = [fr_limbs(a) + fr_limbs(b) for a in pool for b in pool]
    rows += [fr_limbs(rng.randrange(BN_R)) + fr_limbs(rng.randrange(BN_R)) for _ in range(1000)]
    return rows


def cases_fr_cond_sub():
    rng = random.Random(10)
    r = BN_R
    vals = [0, 1, r - 1, r, r + 1, 2 * r - 1, 2 * r - 2]
    vals += [v + d for v in _fr_pool() for d in (0, r)]
    vals += [r + (1 << (64 * j)) for j in range(4)] + [r - (1 << (64 * j)) for j in range(4)]
    vals += [rng.randrange(2 * r) for _ in range(1000)]
    return [fr_limbs(v, 5) for v in vals if 0 <= v < 2 * r]


def cases_fr_canon():
    rng = random.Random(11)
    return [fr_limbs(v) for v in _fr_pool() + [rng.randrange(BN_R) for _ in range(500)]]


CASES = {OP_ACC_REDUCE: cases_acc_reduce, OP_ACC_RUN: cases_acc_run, OP_XACC: cases_xacc, OP_SUB_ADD: cases_sub_add, OP_MUL: cases_mul,
         OP_FOLD: cases_fold, OP_LINE: cases_line, OP_CHAIN: cases_chain, OP_FR: cases_fr, OP_FR_COND_SUB: cases_fr_cond_sub,
         OP_FR_CANON: cases_fr_canon}


# ------------------------------------------------------------------------------------------------ expected outputs
def expect(op, row):
    """The exact outputs of `op` on `row`, in the probe's output order (field elements of BN254 as integers)."""
    if op == OP_ACC_REDUCE:
        return [acc_value(row) % P]
    if op == OP_ACC_RUN:
        x, y, z, reps = row[5:9]
        return [(acc_value(row[:5]) + reps * (x * y + z)) % P]
    if op == OP_XACC:
        x0, x1, y0, y1, yb = row[15:20]
        a00 = acc_value(row[0:5]) + x0 * y0 + x0 * yb
        a11 = acc_value(row[5:10]) + x1 * y1
        ax = acc_value(row[10:15]) + x0 * y1 + x1 * y0 + x1 * yb
        return [(a00 + 7 * a11) % P, ax % P]
    if op == OP_MUL:
        x, y = row[0:2], row[2:4]
        e = ext_mul(x, y)
        return [x[0] * y[0] % P, e[0], e[1], x[0] * y[0] % P, x[1] * y[0] % P, e[0], e[1]]
    if op == OP_FOLD:
        a0, a1, r, c, cr = row[0:2], row[2:4], row[4:6], row[6:8], row[8:10]
        d = ((a1[0] - a0[0]) % P, (a1[1] - a0[1]) % P)
        f = ext_mul(r, d)
        db = (a1[0] - a0[0]) % P
        return [(a0[0] + f[0]) % P, (a0[1] + f[1]) % P, (a0[0] + r[0] * db) % P, r[1] * db % P,
                (c[0] * a0[0] + cr[0] * db) % P, (c[1] * a0[0] + cr[1] * db) % P]
    if op == OP_CHAIN:
        tl, th, ll, lh, rl, rh, q0, q1 = row
        qinf = (lh - ll) * (rh - rl)
        return [x % P for x in (tl * ll * rl, (th - tl) * qinf, (2 * tl - th) * (2 * ll - lh) * (2 * rl - rh), th * lh * rh,
                                tl * q0, (th - tl) * qinf, (2 * tl - th) * (2 * q0 - q1 + 2 * qinf), th * q1)]
    if op == OP_FR:
        a, b = fr_int(row[0:4]), fr_int(row[4:8])
        m = a * b * BN_RINV % BN_R
        return [(a + b) % BN_R, (a - b) % BN_R, m, m]
    if op == OP_FR_COND_SUB:
        return [fr_int(row) % BN_R]
    if op == OP_FR_CANON:
        x = fr_int(row)
        return [x * BN_RM % BN_R, x]
    raise ValueError(op)


def check(op, rows, out):
    """Compare probe output with the exact reference; returns a list of failure descriptions (empty when all agree)."""
    bad = []
    for i, (row, o) in enumerate(zip(rows, out)):
        o = [int(v) for v in o]
        if op == OP_SUB_ADD:
            a, b = row
            ok = (o[0] - (a - b)) % P == 0 and (o[1] - (a + b)) % P == 0 and o[2] == a % P and (a >= P or o[0] < P)
        elif op == OP_LINE:
            lo, hi, q0, q1, qi = row[0:2], row[2:4], row[4], row[5], row[6]
            ok = ((o[0] - (hi[0] - lo[0])) % P == 0 and o[0] < P and (o[1] - (2 * lo[0] - hi[0])) % P == 0
                  and all((o[2 + k] - (hi[k] - lo[k])) % P == 0 and o[2 + k] < P for k in range(2))
                  and all((o[4 + k] - (2 * lo[k] - hi[k])) % P == 0 for k in range(2))
                  and (o[6] - (2 * q0 - q1 + 2 * qi)) % P == 0)
        elif op in (OP_FR, OP_FR_COND_SUB, OP_FR_CANON):
            got = [fr_int(o[4 * k:4 * k + 4]) for k in range(len(o) // 4)]
            ok = got == expect(op, row)
        else:
            want = expect(op, row)
            if op == OP_MUL and not all(v < P for v in row):
                o, want = o[:5], want[:5]          # gl2_mul (the generic product) takes canonical inputs only
            ok = o == want                          # exact: also proves every output canonical
        if not ok:
            bad.append((i, [hex(v) for v in row], [hex(v) for v in o]))
    return bad


# ------------------------------------------------------------------------------------------------ CPU: the tables reach every branch and stay in contract
def test_case_tables_take_every_branch():
    """Every correction branch of the primitives is taken (and not taken) by the committed tables at least a few times, and
    the capacity limits are reached exactly, so a later edit cannot quietly weaken the tables."""
    need = 3

    def both(name, flags):
        n = sum(bool(f) for f in flags)
        assert need <= n <= len(flags) - need, (name, n, len(flags))

    acc = [acc_reduce_branches(s) for s in cases_acc_reduce()]
    both("acc_reduce borrow", [b[0] for b in acc])
    both("acc_reduce carry", [b[1] for b in acc])
    both("acc_reduce canon", [b[2] for b in acc])
    assert all(b[3] <= M32 - 1 for b in acc), "s1 = e3 + 2^32 c must stay canonical"
    assert any(b[3] == M32 - 1 for b in acc), "a state at the e4 limit"
    run = [_run_end_state(r) for r in cases_acc_run()]
    assert all(s[3] <= E4_MAX and s[4] <= M32 for s in run)
    assert sum(s[3] == E4_MAX and s[4] == M32 for s in run) >= need, "runs that end at both capacity limits"
    assert max(r[8] for r in cases_acc_run()) >= (1 << 24) - 1
    sa = cases_sub_add()
    both("gl_sub_cs borrow", [a < b for a, b in sa])
    both("gl_add_cs carry", [a + b > M64 for a, b in sa])
    assert all(b < P for _, b in sa)
    # the line helpers really produce non-canonical values for the chains to consume
    assert any(add_cs(lo, sub_cs(lo, hi)) == P for lo, _, hi, *_ in cases_line())
    assert any(add_cs(r[0], sub_cs(r[0], r[1])) == P for r in cases_chain())
    fr = cases_fr()
    both("fr_sub borrow", [fr_int(r[0:4]) < fr_int(r[4:8]) for r in fr])
    adds = [fr_int(r[0:4]) + fr_int(r[4:8]) for r in fr]
    subs = [fr_int(r) for r in cases_fr_cond_sub()]
    for name, ts in (("fr_cond_sub", subs), ("fr_add", adds)):
        assert sum(t < BN_R for t in ts) >= need, (name, "keep")
        assert sum(t > BN_R for t in ts) >= need, (name, "subtract")
        assert sum(t == BN_R for t in ts) >= 1, (name, "equality")
    assert all(t < 2 * BN_R for t in subs)
    assert all(max(fr_int(r[0:4]), fr_int(r[4:8])) < BN_R for r in fr)
    # every state of the accumulator tables respects its stated capacity
    for s in cases_acc_reduce():
        assert s[3] <= E4_MAX and s[4] <= M32
    for r in cases_xacc():
        for k, room in ((0, 3), (5, 1), (10, 3)):
            assert r[k + 3] <= E4_MAX - room and r[k + 4] <= M32 - 2 * room


def _run_end_state(row):
    """The accumulator state after the run of OP_ACC_RUN, as the device holds it (no column overflows inside the contract)."""
    e01, e23, o01, e4, o2, x, y, z, reps = row
    even = e01 + (e23 << 64) + (e4 << 128) + reps * ((x & M32) * (y & M32) + ((x >> 32) * (y >> 32) << 64) + z)
    odd = o01 + (o2 << 64) + reps * ((x & M32) * (y >> 32) + (x >> 32) * (y & M32))
    assert even >> 160 == 0 and odd >> 96 == 0
    return [even & M64, (even >> 64) & M64, odd & M64, even >> 128, odd >> 64]


def _compile_probe(out_dir):
    from hyper_greco_b200 import build
    so = os.path.join(str(out_dir), "field_probe.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + build.NVCC_FLAGS + ["-I", CSRC, "-o", so, PROBE_SRC]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-4000:]
    return so


def test_probe_compiles_for_sm100a(tmp_path):
    import hyper_greco_b200  # noqa: F401
    so = _compile_probe(tmp_path)
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", so], stdout=subprocess.PIPE, text=True).stdout
    assert "sm_100a" in out
    lib = ctypes.CDLL(so)
    assert lib.probe_run


# ------------------------------------------------------------------------------------------------ GPU: the probe against the references
@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    import hyper_greco_b200  # noqa: F401
    lib = ctypes.CDLL(_compile_probe(tmp_path_factory.mktemp("field_probe")))
    lib.probe_run.restype = ctypes.c_int
    lib.probe_run.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]

    def run(op, rows):
        a = np.ascontiguousarray(np.array(rows, dtype=np.uint64))
        assert a.shape[1] == IN_WORDS[op]
        out = np.zeros((a.shape[0], OUT_WORDS[op]), np.uint64)
        err = lib.probe_run(op, a.ctypes.data, a.shape[1], a.shape[0], out.ctypes.data, out.shape[1])
        assert err == 0, f"CUDA error {err}"
        return out
    return run


OP_NAMES = {OP_ACC_REDUCE: "acc_reduce", OP_ACC_RUN: "acc_mad_add_run", OP_XACC: "xacc", OP_SUB_ADD: "sub_cs_add_cs_canon",
            OP_MUL: "mul_fast", OP_FOLD: "fold", OP_LINE: "slope_at_m1", OP_CHAIN: "gp_chains", OP_FR: "fr_add_sub_mul",
            OP_FR_COND_SUB: "fr_cond_sub", OP_FR_CANON: "fr_canonical_round_trip"}


@pytest.mark.gpu
@pytest.mark.parametrize("op", sorted(OP_NAMES), ids=[OP_NAMES[k] for k in sorted(OP_NAMES)])
def test_device_primitive_matches_exact_arithmetic(probe, op):
    rows = CASES[op]()
    bad = check(op, rows, probe(op, rows))
    assert not bad, f"{OP_NAMES[op]}: {len(bad)} of {len(rows)} cases wrong, first: {bad[:3]}"

