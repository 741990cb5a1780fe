"""BFV SK-encryption witnesses: reference-format loader, synthetic generator, and the Lasso node's input vector.

Host-side tooling (numpy, no GPU). Follows:
  * the witness JSON schema `BfvSkEncryptArgs`            /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:64-73
  * the generator's maths                                 /root/reference/scripts/circuit_sk.py:29-140
  * the input layout `get_inputs`                         /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:365-415
  * the `lasso_inputs_batched` gates and lookup ids       /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:147-210
Coefficient lists are highest degree first, negatives are stored as p - z (circuit_sk.py:155-160).
"""
import json
from dataclasses import dataclass
from typing import List

import numpy as np

from .params import BfvSkEncryptConstants

GL_P = 2**64 - 2**32 + 1
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


@dataclass
class BfvSkEncryptArgs:
    """sk_encryption_circuit.rs:64-73, values as python ints already reduced into [0, p)."""
    s: List[int]
    e: List[int]
    k1: List[int]
    r2is: List[List[int]]
    r1is: List[List[int]]
    ais: List[List[int]]
    ct0is: List[List[int]]


def load_args_json(path) -> BfvSkEncryptArgs:
    d = json.load(open(path))
    cv = lambda v: [int(x) for x in v]
    return BfvSkEncryptArgs(cv(d["s"]), cv(d["e"]), cv(d["k1"]), [cv(v) for v in d["r2is"]], [cv(v) for v in d["r1is"]],
                            [cv(v) for v in d["ais"]], [cv(v) for v in d["ct0is"]])


def dump_args_json(args: BfvSkEncryptArgs, path):
    sv = lambda v: [str(x) for x in v]
    json.dump({"s": sv(args.s), "e": sv(args.e), "k1": sv(args.k1), "r2is": [sv(v) for v in args.r2is],
               "r1is": [sv(v) for v in args.r1is], "ais": [sv(v) for v in args.ais], "ct0is": [sv(v) for v in args.ct0is]}, open(path, "w"))


# ----------------------------------------------------------------------------- synthetic generator
def _conv_ternary_exact(a_obj, s_small):
    """Exact integer product of polynomial a (python ints, |a| < 2^63) with a small-coefficient polynomial s,
    both lowest degree first, via float FFT on 20-bit limbs of a (error << 0.5, see DESIGN.md)."""
    n = len(a_obj)
    size = 1
    while size < 2 * n:
        size <<= 1
    sign = np.array([1 if x >= 0 else -1 for x in a_obj], dtype=np.int64)
    mag = np.array([abs(int(x)) for x in a_obj], dtype=np.uint64)
    fs = np.fft.rfft(np.asarray(s_small, dtype=np.float64), size)
    out = np.zeros(2 * n - 1, dtype=object)
    for limb in range(4):
        part = ((mag >> np.uint64(20 * limb)) & np.uint64((1 << 20) - 1)).astype(np.int64) * sign
        if not part.any():
            continue
        c = np.fft.irfft(np.fft.rfft(part.astype(np.float64), size) * fs, size)[: 2 * n - 1]
        ci = np.rint(c).astype(np.int64)
        assert np.max(np.abs(c - ci)) < 0.05, "FFT convolution lost exactness"
        out = out + ci.astype(object) * (1 << (20 * limb))
    return out


def _center(x, q):
    x %= q
    return x - q if x > (q - 1) // 2 else x


def synth_draws(params: BfvSkEncryptConstants, seed: int):
    """The random part of the synthetic witness (circuit_sk.py:29-70), lowest degree first: s int8, e int8, k1 int32, a [K][n] int64.
    Same generator and the same order of draws as synth_witness, so both describe the same witness."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n, K = params.N, params.K
    s = rng.integers(-1, 2, n)
    e = np.clip(np.rint(rng.normal(0.0, 3.2, n)), -params.E_BOUND, params.E_BOUND).astype(np.int64)
    k1 = rng.integers(-params.K1_BOUND, params.K1_BOUND + 1, n)
    a = np.zeros((K, n), np.int64)
    for i in range(K):
        half = (params.QIS[i] - 1) // 2
        a[i] = rng.integers(-half, half + 1, n, dtype=np.int64)
    return s.astype(np.int8), e.astype(np.int8), k1.astype(np.int32), a


def synth_witness_device(ctx, params: BfvSkEncryptConstants, seed: int):
    """The synthetic witness of synth_witness(params, seed) computed ON THE DEVICE (hg_bfv_witness_generate, csrc/witness_gen.cuh):
    returns (device input buffers in get_inputs / input-node order [s, e, k1, ais.., r1is.., r2is], device buffer of ct0is), in the
    library's representation, ready for Circuit.evaluate and mle_eval_batch."""
    import ctypes as C
    from . import api
    s, e, k1, a = synth_draws(params, seed)
    n, K = params.N, params.K
    eb = 8 * api.LIMBS[ctx.field]
    N2 = 2 * n
    d_s, d_e, d_k1 = (api.DeviceBuffer(ctx, N2 * eb) for _ in range(3))
    d_a, d_r1, d_ct = (api.DeviceBuffer(ctx, K * N2 * eb) for _ in range(3))
    d_r2 = api.DeviceBuffer(ctx, K * n * eb)
    u = lambda v: np.ascontiguousarray(np.array(v[:K], dtype=np.uint64))
    qis, k0is, r1b, r2b = u(params.QIS), u(params.K0IS), u(params.R1_BOUNDS), u(params.R2_BOUNDS)
    vp = lambda x: x.ctypes.data_as(C.c_void_p)
    api._chk(api.lib().hg_bfv_witness_generate(ctx.h, n, K, vp(qis), vp(k0is), vp(r1b), vp(r2b), vp(s), vp(e), vp(k1), vp(np.ascontiguousarray(a)),
                                               d_s.ptr, d_e.ptr, d_k1.ptr, d_a.ptr, d_r1.ptr, d_r2.ptr, d_ct.ptr))
    split = lambda b, cnt, per: [api.DeviceView(b, i * per * eb, per * eb) for i in range(cnt)]
    return [d_s, d_e, d_k1] + split(d_a, K, N2) + split(d_r1, K, N2) + [d_r2], d_ct


def synth_witness(params: BfvSkEncryptConstants, seed: int, p: int = GL_P) -> BfvSkEncryptArgs:
    """Synthetic BFV SK-encryption witness with the reference's distribution (SURVEY.md 8d; circuit_sk.py:29-140):
    s ternary, e ~ N(0, 3.2^2) clipped to +-E_BOUND, k1 uniform in +-K1_BOUND, a_i uniform in +-(q_i-1)/2."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n, K = params.N, params.K
    # lowest degree first internally
    s = rng.integers(-1, 2, n)
    e = np.clip(np.rint(rng.normal(0.0, 3.2, n)), -params.E_BOUND, params.E_BOUND).astype(np.int64)
    k1 = rng.integers(-params.K1_BOUND, params.K1_BOUND + 1, n)
    out = BfvSkEncryptArgs([], [], [], [], [], [], [])
    to_p = lambda v: [int(x) % p for x in v]
    out.s, out.e, out.k1 = to_p(s[::-1]), to_p(e[::-1]), to_p(k1[::-1])
    e_o, k1_o = e.astype(object), k1.astype(object)
    for i in range(K):
        q, k0 = params.QIS[i], params.K0IS[i]
        half = (q - 1) // 2
        a = rng.integers(-half, half + 1, n, dtype=np.int64).astype(object)
        hat = _conv_ternary_exact(a, s)  # degree 2n-2
        hat[:n] = hat[:n] + e_o + k1_o * k0
        red = hat[:n].copy()
        red[: n - 1] = red[: n - 1] - hat[n:]
        ct0 = np.array([_center(int(x), q) for x in red], dtype=object)
        num = -hat
        num[:n] = num[:n] + ct0
        numc = np.array([_center(int(x), q) for x in num], dtype=object)
        r2 = numc[n:]  # degree n-2
        assert all(numc[k] == r2[k] for k in range(n - 1)) and numc[n - 1] == 0, "ct0i - ct0i_hat is not a multiple of x^n+1 mod q"
        rem = num.copy()
        rem[: n - 1] = rem[: n - 1] - r2
        rem[n:] = rem[n:] - r2
        assert all(int(x) % q == 0 for x in rem)
        r1 = np.array([int(x) // q for x in rem], dtype=object)
        assert max(abs(int(x)) for x in r1) <= params.R1_BOUNDS[i], "r1 out of range"
        assert max(abs(int(x)) for x in r2) <= params.R2_BOUNDS[i], "r2 out of range"
        out.ais.append(to_p(a[::-1]))
        out.ct0is.append(to_p(ct0[::-1]))
        out.r2is.append(to_p(r2[::-1]))
        out.r1is.append(to_p(r1[::-1]))
    return out


# ----------------------------------------------------------------------------- input layout
def _padded(v, log2_size):  # poly.rs:21-29
    return list(v) + [0] * ((1 << log2_size) - len(v))


def _shifted(v, size):  # poly.rs:31-44
    pad = max(0, size - len(v))
    out = [0] * pad + list(v)
    np2 = 1
    while np2 < size:
        np2 <<= 1
    return out + [0] * (np2 - len(out))


def get_inputs(params: BfvSkEncryptConstants, args: BfvSkEncryptArgs):
    """sk_encryption_circuit.rs:365-415 -> (dict of input vectors, ct0is output vector), python ints."""
    L, K = params.log2_size, params.K
    s = _padded(args.s, L)
    e = _shifted(args.e, (1 << L) - 1)
    k1 = _shifted(args.k1, (1 << L) - 1)
    r2is, r1is, ais, ct0is = [], [], [], []
    for z in range(min(len(args.ct0is), K)):
        r2is += list(args.r2is[z]) + [0]
        r1is.append(_padded(args.r1is[z], L))
        ais.append(_padded(args.ais[z], L))
        ct = _shifted(args.ct0is[z], 1 << L)[1:] + [0]
        ct0is += ct
    return dict(s=s, e=e, k1=k1, ais=ais, r1is=r1is, r2is=r2is), ct0is


def lasso_lookup_bounds(params: BfvSkEncryptConstants):
    """Bounds of the RangeLookup types handed to LassoPreprocessing::preprocess (sk_encryption_circuit.rs:327-341)."""
    K = params.K
    return ([params.S_BOUND * 2 + 1, params.E_BOUND * 2 + 1, params.K1_BOUND * 2 + 1] + [b * 2 + 1 for b in params.R1_BOUNDS[:K]]
            + [b * 2 + 1 for b in params.R2_BOUNDS[:K]])


def lasso_lookup_segments(params: BfvSkEncryptConstants):
    """The `lookups: Vec<LookupId>` of the Lasso node as (bound, run length) segments (sk_encryption_circuit.rs:182-210)."""
    L, K = params.log2_size, params.K
    r2i_log2 = L if K == 1 else params.N_LOG2
    segs = [(b * 2 + 1, 1 << L) for b in params.R1_BOUNDS[:K]]
    segs += [(b * 2 + 1, 1 << r2i_log2) for b in params.R2_BOUNDS[:K]]
    segs += [(params.S_BOUND * 2 + 1, 1 << L), (params.E_BOUND * 2 + 1, 1 << L), (params.K1_BOUND * 2 + 1, 1 << L)]
    return segs


def lasso_num_vars(params: BfvSkEncryptConstants):
    n = sum(l for _, l in lasso_lookup_segments(params))
    return (n - 1).bit_length()


def lasso_inputs(params: BfvSkEncryptConstants, args: BfvSkEncryptArgs, p: int = GL_P):
    """Output of the `lasso_inputs_batched` VanillaNode (sk_encryption_circuit.rs:163-181): every range-checked
    vector shifted by its bound, concatenated r1is | r2is chunks | s | e | k1. Q7: all r2 chunks use R2_BOUNDS[0]."""
    L, K = params.log2_size, params.K
    ins, _ = get_inputs(params, args)
    size = 1 << L
    r2 = ins["r2is"]
    chunks = [r2[i:i + size] for i in range(0, len(r2), size)]  # sk_encryption_circuit.rs:150-161
    chunks = [c + [0] * (size - len(c)) for c in chunks]
    vecs = [(ins["r1is"][i], params.R1_BOUNDS[i]) for i in range(K)]
    vecs += [(c, params.R2_BOUNDS[0]) for c in chunks]
    vecs += [(ins["s"], params.S_BOUND), (ins["e"], params.E_BOUND), (ins["k1"], params.K1_BOUND)]
    out = []
    for v, b in vecs:
        out += [(x + b) % p for x in v]
    return out


def check_circuit_identity(params: BfvSkEncryptConstants, args: BfvSkEncryptArgs, p: int = GL_P, samples: int = 3, seed: int = 1):
    """ct0i = s*ai + e + k1*k0i + r1i*qi + r2i*(x^n+1) mod p, checked at random evaluation points (Schwartz-Zippel)."""
    import random
    rnd = random.Random(seed)
    n = params.N
    ev = lambda coeffs_hi_first, x: _horner(coeffs_hi_first, x, p)
    for _ in range(samples):
        x = rnd.randrange(p)
        s, e, k1 = ev(args.s, x), ev(args.e, x), ev(args.k1, x)
        for i in range(params.K):
            lhs = ev(args.ct0is[i], x)
            rhs = (s * ev(args.ais[i], x) + e + k1 * params.K0IS[i] + ev(args.r1is[i], x) * params.QIS[i]
                   + ev(args.r2is[i], x) * (pow(x, n, p) + 1)) % p
            if lhs != rhs:
                return False
    return True


def _horner(c, x, p):
    acc = 0
    for v in c:
        acc = (acc * x + v) % p
    return acc


# ----------------------------------------------------------------------------- public-key encryption
# For every modulus i, over Z[x] (params.BfvPkEncryptConstants):
#   ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)
#   ct1_i = pk1_i u + e1           + p1_i q_i + p2_i (x^n + 1)
# The same arithmetic as the SK witness, once per component; the layouts are the SK ones (u as s; e0, e1, k1 as e; pk0is, pk1is as
# ais; r1is, p1is as r1is; r2is, p2is as r2is; ct0is, ct1is as ct0is).
@dataclass
class BfvPkEncryptArgs:
    """Values as python ints already reduced into [0, p), coefficient lists highest degree first."""
    u: List[int]
    e0: List[int]
    e1: List[int]
    k1: List[int]
    pk0is: List[List[int]]
    pk1is: List[List[int]]
    r1is: List[List[int]]
    r2is: List[List[int]]
    p1is: List[List[int]]
    p2is: List[List[int]]
    ct0is: List[List[int]]
    ct1is: List[List[int]]


def synth_pk_draws(params, seed: int):
    """The random part of the synthetic PK witness, lowest degree first, drawn from PCG64(seed) in this order: u (ternary, int8),
    e0, e1 (N(0, 3.2^2) rounded and clipped to +-E_BOUND, int8), k1 (uniform +-K1_BOUND, int32), pk0 [K][n], pk1 [K][n] (uniform
    +-(q_i-1)/2, int64)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n, K = params.N, params.K
    u = rng.integers(-1, 2, n)
    e0 = np.clip(np.rint(rng.normal(0.0, 3.2, n)), -params.E_BOUND, params.E_BOUND).astype(np.int64)
    e1 = np.clip(np.rint(rng.normal(0.0, 3.2, n)), -params.E_BOUND, params.E_BOUND).astype(np.int64)
    k1 = rng.integers(-params.K1_BOUND, params.K1_BOUND + 1, n)
    pk = np.zeros((2, K, n), np.int64)
    for c in range(2):
        for i in range(K):
            half = (params.QIS[i] - 1) // 2
            pk[c, i] = rng.integers(-half, half + 1, n, dtype=np.int64)
    return u.astype(np.int8), e0.astype(np.int8), e1.astype(np.int8), k1.astype(np.int32), pk[0], pk[1]


def _quotients(hat, n, q, q1_bound, q2_bound, what):
    """hat (lowest degree first, 2n-1 coefficients, python ints) -> (ct, q1, q2) with ct = hat + q1 q + q2 (x^n + 1), ct centred
    mod q of degree < n, q1 of degree 2n-2, q2 of degree n-2."""
    red = hat[:n].copy()
    red[: n - 1] = red[: n - 1] - hat[n:]
    ct = np.array([_center(int(x), q) for x in red], dtype=object)
    num = -hat
    num[:n] = num[:n] + ct
    numc = np.array([_center(int(x), q) for x in num], dtype=object)
    q2 = numc[n:]
    assert all(numc[k] == q2[k] for k in range(n - 1)) and numc[n - 1] == 0, f"{what}: not a multiple of x^n+1 mod q"
    rem = num.copy()
    rem[: n - 1] = rem[: n - 1] - q2
    rem[n:] = rem[n:] - q2
    assert all(int(x) % q == 0 for x in rem), f"{what}: not divisible by q"
    q1 = np.array([int(x) // q for x in rem], dtype=object)
    assert max(abs(int(x)) for x in q1) <= q1_bound, f"{what}: first quotient out of range"
    assert max(abs(int(x)) for x in q2) <= q2_bound, f"{what}: second quotient out of range"
    return ct, q1, q2


def synth_pk_witness(params, seed: int, p: int = GL_P) -> BfvPkEncryptArgs:
    """Synthetic BFV PK-encryption witness from synth_pk_draws(params, seed), reduced mod p."""
    u, e0, e1, k1, pk0, pk1 = synth_pk_draws(params, seed)
    n, K = params.N, params.K
    to_p = lambda v: [int(x) % p for x in v]
    out = BfvPkEncryptArgs(to_p(u[::-1]), to_p(e0[::-1]), to_p(e1[::-1]), to_p(k1[::-1]), [], [], [], [], [], [], [], [])
    u_s = u.astype(np.int64)
    e0_o, e1_o, k1_o = e0.astype(object), e1.astype(object), k1.astype(object)
    for i in range(K):
        q = params.QIS[i]
        a0, a1 = pk0[i].astype(object), pk1[i].astype(object)
        hat0 = _conv_ternary_exact(a0, u_s)
        hat0[:n] = hat0[:n] + e0_o + k1_o * params.K0IS[i]
        hat1 = _conv_ternary_exact(a1, u_s)
        hat1[:n] = hat1[:n] + e1_o
        ct0, r1, r2 = _quotients(hat0, n, q, params.R1_BOUNDS[i], params.R2_BOUNDS[i], "ct0")
        ct1, p1, p2 = _quotients(hat1, n, q, params.P1_BOUNDS[i], params.P2_BOUNDS[i], "ct1")
        out.pk0is.append(to_p(a0[::-1]))
        out.pk1is.append(to_p(a1[::-1]))
        out.r1is.append(to_p(r1[::-1]))
        out.r2is.append(to_p(r2[::-1]))
        out.p1is.append(to_p(p1[::-1]))
        out.p2is.append(to_p(p2[::-1]))
        out.ct0is.append(to_p(ct0[::-1]))
        out.ct1is.append(to_p(ct1[::-1]))
    return out


PK_INPUT_NAMES = ("u", "e0", "e1", "k1", "pk0is", "pk1is", "r1is", "p1is", "r2is", "p2is")


def pk_get_inputs(params, args: BfvPkEncryptArgs):
    """-> (dict of input vectors, ct0is, ct1is), python ints. Input-node order: u, e0, e1, k1, pk0is.., pk1is.., r1is.., p1is.., r2is,
    p2is (pk_input_list)."""
    L, K = params.log2_size, params.K
    ins = dict(u=_padded(args.u, L), e0=_shifted(args.e0, (1 << L) - 1), e1=_shifted(args.e1, (1 << L) - 1), k1=_shifted(args.k1, (1 << L) - 1))
    for key in ("pk0is", "pk1is", "r1is", "p1is"):
        ins[key] = [_padded(v, L) for v in getattr(args, key)[:K]]
    for key in ("r2is", "p2is"):
        ins[key] = [x for v in getattr(args, key)[:K] for x in list(v) + [0]]
    cts = [[x for v in getattr(args, key)[:K] for x in _shifted(v, 1 << L)[1:] + [0]] for key in ("ct0is", "ct1is")]
    return ins, cts[0], cts[1]


def pk_input_list(ins):
    """The dict of pk_get_inputs as the list of input-node vectors, insertion order."""
    return [ins["u"], ins["e0"], ins["e1"], ins["k1"]] + list(ins["pk0is"]) + list(ins["pk1is"]) + list(ins["r1is"]) + list(ins["p1is"]) + \
        [ins["r2is"], ins["p2is"]]


def pk_lasso_lookup_bounds(params):
    """Bounds (2b + 1) of the range lookups of the PK circuit's Lasso preprocessing; equal bounds are one lookup type."""
    K = params.K
    return ([params.U_BOUND * 2 + 1, params.E_BOUND * 2 + 1, params.K1_BOUND * 2 + 1] + [b * 2 + 1 for b in params.R1_BOUNDS[:K]]
            + [b * 2 + 1 for b in params.P1_BOUNDS[:K]] + [b * 2 + 1 for b in params.R2_BOUNDS[:K]] + [b * 2 + 1 for b in params.P2_BOUNDS[:K]])


def pk_lasso_lookup_segments(params):
    """The Lasso node's lookups as (bound, run length) segments, in the order of its input layer: r1is, p1is, r2 chunks, p2 chunks,
    u, e0, e1, k1. A quotient of the second kind has n rows per modulus (2n for K = 1, padding included)."""
    L, K = params.log2_size, params.K
    q2_len = 1 << (L if K == 1 else params.N_LOG2)
    segs = [(b * 2 + 1, 1 << L) for b in params.R1_BOUNDS[:K]]
    segs += [(b * 2 + 1, 1 << L) for b in params.P1_BOUNDS[:K]]
    segs += [(b * 2 + 1, q2_len) for b in params.R2_BOUNDS[:K]]
    segs += [(b * 2 + 1, q2_len) for b in params.P2_BOUNDS[:K]]
    segs += [(b * 2 + 1, 1 << L) for b in (params.U_BOUND, params.E_BOUND, params.E_BOUND, params.K1_BOUND)]
    return segs


def pk_lasso_num_vars(params):
    n = sum(l for _, l in pk_lasso_lookup_segments(params))
    return (n - 1).bit_length()


def pk_lasso_inputs(params, args: BfvPkEncryptArgs, p: int = GL_P):
    """The values of the Lasso node's input layer: every range-checked element shifted by the bound of its own vector, concatenated
    r1is | p1is | r2 chunks | p2 chunks | u | e0 | e1 | k1. A chunk element at flat index f belongs to modulus f / n (modulus 0 for
    the zero padding of K = 1)."""
    L, K, n = params.log2_size, params.K, params.N
    ins, _, _ = pk_get_inputs(params, args)
    size = 1 << L
    out = []

    def shifted(v, bounds_of):
        out.extend((x + bounds_of(j)) % p for j, x in enumerate(v))
    for key, bounds in (("r1is", params.R1_BOUNDS), ("p1is", params.P1_BOUNDS)):
        for i in range(K):
            shifted(ins[key][i], lambda j, b=bounds[i]: b)
    for key, bounds in (("r2is", params.R2_BOUNDS), ("p2is", params.P2_BOUNDS)):
        v = list(ins[key])
        v += [0] * ((-len(v)) % size)
        shifted(v, lambda f, b=bounds: b[min(f // n, K - 1)])
    for key, b in (("u", params.U_BOUND), ("e0", params.E_BOUND), ("e1", params.E_BOUND), ("k1", params.K1_BOUND)):
        shifted(ins[key], lambda j, b=b: b)
    return out


def check_pk_circuit_identity(params, args: BfvPkEncryptArgs, p: int = GL_P, samples: int = 3, seed: int = 1):
    """Both relations mod p at random evaluation points (Schwartz-Zippel)."""
    import random
    rnd = random.Random(seed)
    n = params.N
    for _ in range(samples):
        x = rnd.randrange(p)
        ev = lambda c: _horner(c, x, p)
        u, e0, e1, k1 = ev(args.u), ev(args.e0), ev(args.e1), ev(args.k1)
        cyclo = (pow(x, n, p) + 1) % p
        for i in range(params.K):
            q = params.QIS[i]
            if ev(args.ct0is[i]) != (ev(args.pk0is[i]) * u + e0 + k1 * params.K0IS[i] + ev(args.r1is[i]) * q + ev(args.r2is[i]) * cyclo) % p:
                return False
            if ev(args.ct1is[i]) != (ev(args.pk1is[i]) * u + e1 + ev(args.p1is[i]) * q + ev(args.p2is[i]) * cyclo) % p:
                return False
    return True


def synth_pk_witness_device(ctx, params, seed: int):
    """The witness of synth_pk_witness(params, seed) computed on the device (hg_bfv_pk_witness_generate): returns (device input
    buffers in input-node order [u, e0, e1, k1, pk0is.., pk1is.., r1is.., p1is.., r2is, p2is], d_ct0is, d_ct1is) in the library's
    representation."""
    return pk_witness_device_from_draws(ctx, params, *synth_pk_draws(params, seed))


def pk_witness_device_from_draws(ctx, params, u, e0, e1, k1, pk0, pk1):
    import ctypes as C
    from . import api
    n, K = params.N, params.K
    eb = 8 * api.LIMBS[ctx.field]
    N2 = 2 * n
    small = [api.DeviceBuffer(ctx, N2 * eb) for _ in range(4)]
    wide = [api.DeviceBuffer(ctx, K * N2 * eb) for _ in range(4)]      # pk0is, pk1is, r1is, p1is
    narrow = [api.DeviceBuffer(ctx, K * n * eb) for _ in range(2)]     # r2is, p2is
    d_ct0, d_ct1 = api.DeviceBuffer(ctx, K * N2 * eb), api.DeviceBuffer(ctx, K * N2 * eb)
    arr = lambda v: np.ascontiguousarray(np.array(v[:K], dtype=np.uint64))
    keep = [arr(params.QIS), arr(params.K0IS), arr(params.R1_BOUNDS), arr(params.R2_BOUNDS), arr(params.P1_BOUNDS), arr(params.P2_BOUNDS),
            np.ascontiguousarray(u, np.int8), np.ascontiguousarray(e0, np.int8), np.ascontiguousarray(e1, np.int8), np.ascontiguousarray(k1, np.int32),
            np.ascontiguousarray(pk0, np.int64), np.ascontiguousarray(pk1, np.int64)]
    vp = lambda x: x.ctypes.data_as(C.c_void_p)
    api._chk(api.lib().hg_bfv_pk_witness_generate(ctx.h, n, K, *[vp(x) for x in keep], *[b.ptr for b in small + wide + narrow + [d_ct0, d_ct1]]))
    split = lambda b, cnt, per: [api.DeviceView(b, i * per * eb, per * eb) for i in range(cnt)]
    return small + [v for b in wide for v in split(b, K, N2)] + narrow, d_ct0, d_ct1
