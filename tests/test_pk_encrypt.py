"""BFV public-key encryption: parameters, witness, circuit, prover and verifiers.

For every modulus i < K over Z[x]:  ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1),  ct1_i = pk1_i u + e1 + p1_i q_i + p2_i (x^n + 1).
On the CPU: the parameter derivation, the numpy witness, the CPU restatement of the circuit (tests/pk_encrypt_oracle.cpp, on the
oracle) proving and verifying, the library's host verifier accepting the restatement's proofs with the same input claims, and both
verifiers rejecting tampered proofs and statements. On the GPU (-m gpu): the device witness generator against numpy, device
evaluation, proof bytes and input claims against the restatement in every schedule and at full size, a sharded proof, and batched
verification against the host verifier."""
import ctypes as C
import gc
import hashlib
import os

import numpy as np
import pytest

GL_P = 2**64 - 2**32 + 1
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
PRIME = {0: GL_P, 1: BN_R}
SMALL_CASES = [pytest.param(0, "1024_1x27_65537", id="goldilocks-1024"), pytest.param(1, "1024_1x27_65537", id="bn254-1024"),
               pytest.param(0, "4096_2x55_65537", id="goldilocks-4096")]


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, build
    build.build()
    api.lib()
    return api


# ------------------------------------------------------------------------------------------------ CPU restatement
# tests/pk_encrypt_oracle.cpp, compiled with g++ into the temporary directory (the tree may be read-only), once per source version.
_PKLIB = None


def _pklib():
    global _PKLIB
    if _PKLIB is None:
        import subprocess
        import tempfile
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        src = os.path.join(root, "tests", "pk_encrypt_oracle.cpp")
        deps = [src] + [os.path.join(root, "oracle", f) for f in sorted(os.listdir(os.path.join(root, "oracle"))) if f.endswith(".hpp")]
        tag = hashlib.sha256(b"".join(open(d, "rb").read() for d in deps)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"hg_pk_encrypt_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.check_call([cxx, "-O3", "-march=x86-64-v3", "-std=c++17", "-fopenmp", "-fPIC", "-shared", "-w",
                                   "-I", os.path.join(root, "oracle"), "-o", tmp, src])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp, sz, u64 = C.c_void_p, C.c_size_t, C.c_uint64
        L.hgpk_last_error.restype = C.c_char_p
        L.hgpk_new.argtypes = [C.c_int, C.c_int, C.c_int, vp, u64, u64, u64, C.POINTER(vp)]
        L.hgpk_free.argtypes = [vp]
        L.hgpk_set_assumption.argtypes = [C.c_int, C.c_int]
        L.hgpk_lasso_num_vars.argtypes = [vp]
        L.hgpk_evaluate.argtypes = [vp, vp]
        L.hgpk_value.argtypes = [vp, C.c_int, vp, C.POINTER(sz)]
        L.hgpk_prove.argtypes = [vp, vp, vp, vp, sz, C.POINTER(sz)]
        L.hgpk_verify.argtypes = [vp, vp, vp, vp, vp, sz]
        L.hgpk_num_inputs.restype = sz
        L.hgpk_num_inputs.argtypes = [vp]
        L.hgpk_num_claims.restype = sz
        L.hgpk_num_claims.argtypes = [vp, sz]
        L.hgpk_claim.argtypes = [vp, sz, sz, vp, vp, C.POINTER(sz)]
        _PKLIB = L
    return _PKLIB


class RestatementError(RuntimeError):
    pass


def _gp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _chk(rc):
    if rc != 0:
        raise RestatementError(_pklib().hgpk_last_error().decode())


class PkRestatement:
    """The PK circuit on the CPU restatement: evaluate / prove / verify; vectors are canonical limb arrays."""

    def __init__(self, field, P):
        self.field, self.P, self.limbs = field, P, 1 if field == 0 else 4
        K = P.K
        b = np.ascontiguousarray(np.concatenate([np.array(v[:K], np.uint64) for v in (P.QIS, P.K0IS, P.R1_BOUNDS, P.R2_BOUNDS, P.P1_BOUNDS, P.P2_BOUNDS)]))
        self.h = C.c_void_p()
        _chk(_pklib().hgpk_new(field, P.log2_size, K, _gp(b), P.U_BOUND, P.E_BOUND, P.K1_BOUND, C.byref(self.h)))

    @property
    def lasso_num_vars(self):
        return int(_pklib().hgpk_lasso_num_vars(self.h))

    @staticmethod
    def _cat(vecs):
        return np.ascontiguousarray(np.concatenate([np.asarray(v, np.uint64).reshape(-1) for v in vecs]))

    def evaluate(self, inputs):
        self._keep = self._cat(inputs)
        _chk(_pklib().hgpk_evaluate(self.h, _gp(self._keep)))

    def value(self, which):
        """0: the Lasso node's input layer, 1: sum0, 2: sum1"""
        n = C.c_size_t(0)
        _chk(_pklib().hgpk_value(self.h, which, None, C.byref(n)))
        out = np.zeros(n.value * self.limbs, np.uint64)
        _chk(_pklib().hgpk_value(self.h, which, _gp(out), C.byref(n)))
        return out

    def prove(self, ct0, ct1):
        c0, c1 = self._cat([ct0]), self._cat([ct1])
        n = C.c_size_t(0)
        buf = np.zeros(1 << 24, np.uint8)
        _chk(_pklib().hgpk_prove(self.h, _gp(c0), _gp(c1), _gp(buf), buf.size, C.byref(n)))
        assert n.value <= buf.size
        return buf[: n.value].tobytes(), self._claims()

    def verify(self, inputs, ct0, ct1, proof):
        ins, c0, c1 = self._cat(inputs), self._cat([ct0]), self._cat([ct1])
        buf = np.frombuffer(proof, np.uint8).copy() if proof else np.zeros(1, np.uint8)
        _chk(_pklib().hgpk_verify(self.h, _gp(ins), _gp(c0), _gp(c1), _gp(buf), len(proof)))
        return self._claims()

    def _claims(self):
        el = self.limbs * (2 if self.field == 0 else 1)
        L = _pklib()
        out = []
        for i in range(L.hgpk_num_inputs(self.h)):
            cl = []
            for k in range(L.hgpk_num_claims(self.h, i)):
                nv = C.c_size_t(0)
                _chk(L.hgpk_claim(self.h, i, k, None, None, C.byref(nv)))
                pt, v = np.zeros((nv.value, el), np.uint64), np.zeros(el, np.uint64)
                _chk(L.hgpk_claim(self.h, i, k, _gp(pt), _gp(v), C.byref(nv)))
                cl.append((pt, v))
            out.append(cl)
        return out

    def __del__(self):
        try:
            if self.h:
                _pklib().hgpk_free(self.h)
                self.h = None
        except Exception:
            pass


def limbs(vals, field):
    vals = [int(x) for x in vals]
    if field == 0:
        return np.array(vals, dtype=np.uint64)
    out = np.zeros(len(vals) * 4, np.uint64)
    for i, v in enumerate(vals):
        for j in range(4):
            out[4 * i + j] = (v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF
    return out


_INSTANCES = {}


def instance(field, name, seed=1):
    """(P, args, host input limbs in input-node order, ct0 limbs, ct1 limbs) of the numpy witness"""
    key = (field, name, seed)
    if key not in _INSTANCES:
        from hyper_greco_b200 import params, witness
        P = params.PK_PARAMS[name]
        args = witness.synth_pk_witness(P, seed, PRIME[field])
        ins, ct0, ct1 = witness.pk_get_inputs(P, args)
        _INSTANCES[key] = (P, args, [limbs(v, field) for v in witness.pk_input_list(ins)], limbs(ct0, field), limbs(ct1, field))
    return _INSTANCES[key]


_PROOFS = {}


def restatement_proof(field, name, seed=1):
    """the restatement's (proof, input claims) of instance(field, name, seed), proved once"""
    key = (field, name, seed)
    if key not in _PROOFS:
        P, _, flat, ct0, ct1 = instance(field, name, seed)
        r = PkRestatement(field, P)
        r.evaluate(flat)
        _PROOFS[key] = r.prove(ct0, ct1)
    return _PROOFS[key]


def same_claims(a, b):
    return len(a) == len(b) and all(len(x) == len(y) and all((p == q).all() and (v == w).all() for (p, v), (q, w) in zip(x, y)) for x, y in zip(a, b))


def claims_match_inputs(api, field, inputs, claims):
    return all((api.mle_eval_host(field, vec, pt.shape[0], pt) == v).all() for vec, cl in zip(inputs, claims) for pt, v in cl) and all(claims)


# ------------------------------------------------------------------------------------------------ CPU
def test_pk_params_follow_the_sk_sets(api):
    """floor((n h U + E + K1 k0_i + 2h) / q_i), h = (q_i - 1) / 2, reproduces every SK R1 bound, so the same rule without the k1 term
    bounds P1; every PK set is derived from its SK set."""
    from hyper_greco_b200 import params
    checked = 0
    for sk in params.PARAMS.values():
        for i, q in enumerate(sk.QIS):
            assert params.quotient_bound(sk.N, q, sk.S_BOUND, sk.E_BOUND, sk.K1_BOUND * sk.K0IS[i]) == sk.R1_BOUNDS[i]
            checked += 1
    assert checked == sum(p.K for p in params.PARAMS.values())
    assert set(params.PK_PARAMS) == set(params.PARAMS)
    for name, sk in params.PARAMS.items():
        pk = params.PK_PARAMS[name]
        assert (pk.name, pk.N, pk.QIS, pk.K0IS, pk.E_BOUND, pk.K1_BOUND) == (name, sk.N, sk.QIS, sk.K0IS, sk.E_BOUND, sk.K1_BOUND)
        assert pk.U_BOUND == sk.S_BOUND and pk.K == sk.K and pk.log2_size == sk.log2_size
        assert pk.R1_BOUNDS == sk.R1_BOUNDS and pk.R2_BOUNDS == pk.P2_BOUNDS == sk.R2_BOUNDS
        for i, q in enumerate(sk.QIS):
            h = (q - 1) // 2
            assert pk.P1_BOUNDS[i] == (sk.N * h * sk.S_BOUND + sk.E_BOUND + 2 * h) // q


@pytest.mark.parametrize("name", ["1024_1x27_65537", "2048_1x52_65537", "4096_2x55_65537"])
def test_numpy_pk_witness_satisfies_both_relations(api, name):
    from hyper_greco_b200 import params, witness
    P = params.PK_PARAMS[name]
    args = witness.synth_pk_witness(P, 3)
    assert witness.check_pk_circuit_identity(P, args)
    bad = witness.BfvPkEncryptArgs(**{**args.__dict__, "ct1is": [[(x + 1) % GL_P for x in args.ct1is[0]]] + args.ct1is[1:]})
    assert not witness.check_pk_circuit_identity(P, bad)
    rows = [b for b, l in witness.pk_lasso_lookup_segments(P) for _ in range(l)]   # every shifted element lies in its table [0, 2b + 1)
    lasso_in = witness.pk_lasso_inputs(P, args)
    assert len(rows) == len(lasso_in) and all(x < b for x, b in zip(lasso_in, rows))


@pytest.mark.parametrize("field,name", SMALL_CASES)
def test_restatement_proves_and_verifies(api, field, name):
    from hyper_greco_b200 import witness
    P, args, flat, ct0, ct1 = instance(field, name)
    r = PkRestatement(field, P)
    assert r.lasso_num_vars == witness.pk_lasso_num_vars(P)
    r.evaluate(flat)
    assert (r.value(1) == ct0).all() and (r.value(2) == ct1).all()
    lasso_in, want = r.value(0), limbs(witness.pk_lasso_inputs(P, args, PRIME[field]), field)   # the layer is padded to a power of two
    assert (lasso_in[: want.size] == want).all() and not lasso_in[want.size:].any()
    proof, claims = restatement_proof(field, name)
    assert same_claims(r.verify(flat, ct0, ct1, proof), claims)
    assert claims_match_inputs(api, field, flat, claims)
    # the library's host verifier accepts it with the same input claims
    assert same_claims(api.BfvPkEncryptVerifier(P, field).verify(flat, ct0, ct1, proof), claims)


def tamper_cases(api, field, name):
    """(label, inputs, ct0, ct1, proof) statements that both verifiers must reject. Proof elements are located by replaying the
    host verifier through a logging transcript: sum1 is proved first, then sum0 (it starts after sum1's four input evaluations), the
    Lasso node starts with the first read after its lasso_num_vars squeezes."""
    from hyper_greco_b200 import witness
    P, _, flat, ct0, ct1 = instance(field, name)
    proof, _ = restatement_proof(field, name)
    v = api.BfvPkEncryptVerifier(P, field)
    tr = api.CallbackTranscript(api.Keccak256Transcript.from_proof(proof, field), field)
    L = v.ct_log2_size
    pts = [tr.squeeze_challenges(L), tr.squeeze_challenges(L)]
    vals = [api.mle_eval_host(field, c, L, p) for c, p in zip((ct0, ct1), pts)]
    v.circuit.verify_gkr(api._pk_output_claims(pts[0], vals[0], pts[1], vals[1]), tr)
    kinds = [k for k, _ in tr.log][2 * L:]
    reads_before, groups, nread, run, lasso_at = [], [], 0, 0, None
    for k in kinds:                          # groups of consecutive reads: (first read index, length)
        if k == "read":
            if run >= witness.pk_lasso_num_vars(P) and lasso_at is None:
                lasso_at = nread
            if not groups or reads_before[-1] != "read":
                groups.append([nread, 0])
            groups[-1][1] += 1
            nread += 1
            run = 0
        else:
            run += 1
        reads_before.append(k)
    esz = 8 * (1 if field == 0 else 4) * (2 if field == 0 else 1)
    assert nread * esz == len(proof) and lasso_at is not None
    sum0_at = next(g[0] for g in groups if g[1] > 2) + 4
    assert groups[0][0] == 0 and sum0_at < lasso_at

    def flip(elem):
        bsz = 8 * (1 if field == 0 else 4)
        off = elem * esz
        x = (int.from_bytes(proof[off:off + bsz], "big") + 1) % PRIME[field]
        return proof[:off] + x.to_bytes(bsz, "big") + proof[off + bsz:]
    ct1_bad = ct1.copy()
    lim = 1 if field == 0 else 4
    ct1_bad[(ct1.size // (2 * lim)) * lim] ^= 1
    pk1_bad = [x.copy() for x in flat]
    pk1_bad[4 + P.K][3 * (1 if field == 0 else 4)] ^= 1
    return [("sum1 sumcheck", flat, ct0, ct1, flip(1)), ("sum0 sumcheck", flat, ct0, ct1, flip(sum0_at + 1)),
            ("lasso node", flat, ct0, ct1, flip(lasso_at)), ("last element", flat, ct0, ct1, flip(nread - 1)),
            ("truncated", flat, ct0, ct1, proof[:-esz]), ("trailing byte", flat, ct0, ct1, proof + b"\x00"),
            ("ct1 coefficient", flat, ct0, ct1_bad, proof), ("pk1 coefficient", pk1_bad, ct0, ct1, proof),
            ("ct0 and ct1 swapped", flat, ct1, ct0, proof)]


@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
def test_both_verifiers_reject_tampering(api, field):
    name = "1024_1x27_65537"
    P = instance(field, name)[0]
    r = PkRestatement(field, P)
    v = api.BfvPkEncryptVerifier(P, field)
    for _, ins, c0, c1, pr in tamper_cases(api, field, name):
        with pytest.raises(RestatementError):
            r.verify(ins, c0, c1, pr)
        with pytest.raises(api.HgError):
            v.verify(ins, c0, c1, pr)


def test_configure_rejects_bad_arguments(api):
    from hyper_greco_b200 import params, witness
    P = params.PK_PARAMS["4096_2x55_65537"]
    a = lambda v: np.ascontiguousarray(np.array(v, np.uint64))
    arrs = [a(P.QIS), a(P.K0IS), a(P.R1_BOUNDS), a(P.R2_BOUNDS), a(P.P1_BOUNDS), a(P.P2_BOUNDS)]
    pp = api.LassoPreprocessing.preprocess(witness.pk_lasso_lookup_bounds(P))
    nv = witness.pk_lasso_num_vars(P)

    def call(K=2, nulls=(), lasso=True):
        c = api.Circuit(None, 0)
        ptrs = [None if i in nulls else _gp(x) for i, x in enumerate(arrs)]
        rc = api.lib().hg_bfv_pk_configure(c.h, P.log2_size, K, *ptrs, P.U_BOUND, P.E_BOUND, P.K1_BOUND, None, pp.h if lasso else None, nv, None)
        return rc, api.lib().hg_last_error().decode()
    assert call()[0] == 0
    for i in range(6):
        rc, msg = call(nulls=(i,))
        assert rc != 0 and "hg_bfv_pk_configure" in msg
    rc, msg = call(K=3)
    assert rc != 0 and "power of two" in msg
    rc, msg = call(lasso=False)
    assert rc != 0 and "Lasso" in msg
    assert api.lib().hg_bfv_pk_configure(None, P.log2_size, 2, *[_gp(x) for x in arrs], 1, 19, 1, None, pp.h, nv, None) != 0


def test_pk_witness_generate_needs_a_device(api):
    """The generator refuses NULL arguments with an error, never a crash; without a device no context can be made."""
    L = api.lib()
    assert L.hg_bfv_pk_witness_generate(None, 1024, 1, *([None] * 24)) != 0
    assert "hg_bfv_pk_witness_generate" in L.hg_last_error().decode()
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if not has_gpu:
        with pytest.raises(api.HgError):
            api.Context(0)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctxs(api):
    c = {0: api.Context(0, api.GOLDILOCKS), 1: api.Context(0, api.BN254)}
    yield c
    gc.collect()  # provers and verifiers go before the contexts they were made on
    for x in c.values():
        x.close()


def download(ctx, buf, count):
    return buf.to_field(count).reshape(-1)


def device_limbs(ctx, dev, d_ct0, d_ct1, P):
    """host canonical limbs of a device witness (input-node order), ct0is, ct1is"""
    sizes = [2 * P.N] * 4 + [2 * P.N] * (4 * P.K) + [P.K * P.N] * 2
    return [download(ctx, b, s) for b, s in zip(dev, sizes)], download(ctx, d_ct0, 2 * P.N * P.K), download(ctx, d_ct1, 2 * P.N * P.K)


@pytest.mark.gpu
@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
@pytest.mark.parametrize("name", ["1024_1x27_65537", "2048_1x52_65537", "4096_2x55_65537"])
def test_device_witness_equals_numpy(api, ctxs, field, name):
    from hyper_greco_b200 import witness
    P, _, flat, ct0, ct1 = instance(field, name, seed=2)
    dev, d_ct0, d_ct1 = witness.synth_pk_witness_device(ctxs[field], P, 2)
    got, g0, g1 = device_limbs(ctxs[field], dev, d_ct0, d_ct1, P)
    assert len(got) == len(flat)
    for k, (a, b) in enumerate(zip(got, flat)):
        assert (a == b).all(), k
    assert (g0 == ct0).all() and (g1 == ct1).all()


def args_from_layout(P, host, ct0, ct1):
    """BfvPkEncryptArgs (highest degree first) back from the input layout of a witness (Goldilocks limbs)"""
    from hyper_greco_b200 import witness
    n, K = P.N, P.K
    L = lambda v: [int(x) for x in v]
    sh = lambda v: L(v[n - 1: 2 * n - 1])
    per = lambda base: [host[base + i] for i in range(K)]
    q2 = lambda v: [L(v[i * n: i * n + n - 1]) for i in range(K)]
    cts = lambda c: [sh(c[i * 2 * n: (i + 1) * 2 * n]) for i in range(K)]
    return witness.BfvPkEncryptArgs(
        u=L(host[0][:n]), e0=sh(host[1]), e1=sh(host[2]), k1=sh(host[3]),
        pk0is=[L(v[:n]) for v in per(4)], pk1is=[L(v[:n]) for v in per(4 + K)], r1is=[L(v[:2 * n - 1]) for v in per(4 + 2 * K)],
        p1is=[L(v[:2 * n - 1]) for v in per(4 + 3 * K)], r2is=q2(host[4 + 4 * K]), p2is=q2(host[5 + 4 * K]), ct0is=cts(ct0), ct1is=cts(ct1))


@pytest.mark.gpu
def test_device_witness_full_size_and_bound_errors(api, ctxs):
    """n = 32768, K = 16: the downloaded device witness satisfies both relations; draws that push a quotient past its bound are an
    error that names the component and the quotient."""
    from hyper_greco_b200 import params, witness
    P = params.PK_PARAMS["32768_16x59_65537"]
    ctx = ctxs[0]
    dev, d_ct0, d_ct1 = witness.synth_pk_witness_device(ctx, P, 11)
    host, c0, c1 = device_limbs(ctx, dev, d_ct0, d_ct1, P)
    args = args_from_layout(P, host, c0, c1)
    assert witness.check_pk_circuit_identity(P, args)
    bad = witness.BfvPkEncryptArgs(**{**args.__dict__, "p2is": [[(x + 1) % GL_P for x in args.p2is[0]]] + args.p2is[1:]})
    assert not witness.check_pk_circuit_identity(P, bad)
    Ps = params.PK_PARAMS["1024_1x27_65537"]
    u, e0, e1, k1, pk0, pk1 = witness.synth_pk_draws(Ps, 1)
    u[:] = 1
    big = np.full_like(pk1, Ps.QIS[0] - 1)          # |pk1 u| reaches n (q - 1): p1 near n, twice its bound; ct0 is untouched
    with pytest.raises(api.HgError, match=r"ct1: .*p1 coefficients out of range"):
        witness.pk_witness_device_from_draws(ctx, Ps, u, e0, e1, k1, pk0, big)
    with pytest.raises(api.HgError, match=r"ct0: .*r1 coefficients out of range"):
        witness.pk_witness_device_from_draws(ctx, Ps, u, e0, e1, k1, big, pk1)
    u[0] = 2
    with pytest.raises(api.HgError, match="ternary"):
        witness.pk_witness_device_from_draws(ctx, Ps, u, e0, e1, k1, pk0, pk1)
    witness.synth_pk_witness_device(ctx, Ps, 1)      # the context still works


class Absorbing:
    """A caller transcript whose squeeze hashes everything written or read so far: every proof gets its own points."""

    def __init__(self, field, seed, proof=None):
        self.field, self.state, self.out, self.proof, self.pos = field, hashlib.sha256(b"seed%d" % seed).digest(), [], proof, 0
        self.el = 2 if field == 0 else 4

    def squeeze_challenge(self):
        self.state = hashlib.sha256(self.state + b"squeeze").digest()
        if self.field == 0:
            return np.array([int.from_bytes(self.state[8 * i: 8 * i + 8], "little") % GL_P for i in range(2)], np.uint64)
        v = int.from_bytes(self.state, "little") % BN_R
        return np.array([(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)], np.uint64)

    def write_felt_ext(self, v):
        v = np.asarray(v, np.uint64)
        self.out.append(v.copy())
        self.state = hashlib.sha256(self.state + v.tobytes()).digest()

    def read_felt_ext(self):
        if self.pos + self.el > len(self.proof):
            raise EOFError
        v = self.proof[self.pos: self.pos + self.el]
        self.pos += self.el
        self.state = hashlib.sha256(self.state + v.tobytes()).digest()
        return v

    def into_proof(self):
        return np.concatenate(self.out) if self.out else np.zeros(0, np.uint64)


def _node_values(api, ctx, prover, field):
    out = []
    for key in ("lasso_in", "sum0", "sum1"):
        ptr, n = prover.circuit.node_value(prover.ids[key])
        v = api.NodeValueView(ctx, ptr, n).download(np.uint64, n * (1 if field == 0 else 4))
        if field == 1:
            tmp = api.DeviceBuffer.from_numpy(ctx, v)
            v = tmp.to_field(n).reshape(-1)
        out.append(v)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("field,name", SMALL_CASES)
def test_device_proof_equals_restatement_in_every_schedule(api, ctxs, field, name):
    P, _, flat, ct0, ct1 = instance(field, name)
    want, wclaims = restatement_proof(field, name)
    r = PkRestatement(field, P)
    r.evaluate(flat)
    ctx = ctxs[field]
    prover = api.BfvPkEncryptProver(ctx, P)
    for mode in (api.MODE_PREFETCH, api.MODE_INTERACTIVE):
        proof, claims = prover.prove_host(flat, ct0, ct1, mode)
        assert proof == want, mode
        assert same_claims(claims, wclaims)
        if mode == api.MODE_PREFETCH:
            got = _node_values(api, ctx, prover, field)
            assert all(g.size == r.value(w).size and (g == r.value(w)).all() for g, w in zip(got, (0, 1, 2)))
    for independent in (True, False):        # a caller-owned transcript: message-independent (prefetched) and absorbing (interactive)
        tr = api.CallbackTranscript(api.Keccak256Transcript(field), field, message_independent=independent)
        proof, claims = prover.prove_host(flat, ct0, ct1, api.MODE_PREFETCH, transcript=tr)
        assert proof == want and same_claims(claims, wclaims)
    # device-resident inputs give the same proof
    d_in = [api.DeviceBuffer.from_numpy(ctx, x) for x in flat]
    d_ct = [api.DeviceBuffer.from_numpy(ctx, x) for x in (ct0, ct1)]
    if field == 1:
        for b, x in zip(d_in + d_ct, flat + [ct0, ct1]):
            api._chk(api.lib().hg_field_encode(ctx.h, b.ptr, x.size // 4))
    proof, _ = prover.prove(d_in, d_ct[0], d_ct[1])
    assert proof == want


@pytest.mark.gpu
def test_device_proof_under_non_default_switches(api):
    """A3 evaluations wire format, A3' h(1) from the tables, A5 descending powers: device bytes == restatement bytes, and the host
    verifier accepts with the matching options."""
    field, name = 0, "1024_1x27_65537"
    P, _, flat, ct0, ct1 = instance(field, name)
    opts = {api.OPT_A3_WIRE: 1, api.OPT_A3_H1: 1, api.OPT_A5_ASCENDING: 0}
    ctx = api.Context(0, api.GOLDILOCKS)
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
            _pklib().hgpk_set_assumption(k, v)
        r = PkRestatement(field, P)
        r.evaluate(flat)
        want, wclaims = r.prove(ct0, ct1)
        prover = api.BfvPkEncryptProver(ctx, P)
        proof, claims = prover.prove_host(flat, ct0, ct1)
        assert proof == want and same_claims(claims, wclaims)
        assert proof != restatement_proof(field, name)[0]
        api.BfvPkEncryptVerifier(P).verify(flat, ct0, ct1, proof, [1, 1, 0])
        prover.circuit.free()
        prover.lasso.free()
    finally:
        _pklib().hgpk_set_assumption(3, 0)
        _pklib().hgpk_set_assumption(31, 0)
        _pklib().hgpk_set_assumption(5, 1)
        ctx.close()


@pytest.mark.gpu
def test_two_rank_sharded_proof_equals_single_device(api, ctxs):
    import torch
    field, name = 0, "4096_2x55_65537"
    P, _, flat, ct0, ct1 = instance(field, name)
    ctx = ctxs[0]
    prover = api.BfvPkEncryptProver(ctx, P)
    want, wclaims = prover.prove_host(flat, ct0, ct1)
    d_ct = [api.DeviceBuffer.from_numpy(ctx, x) for x in (ct0, ct1)]
    L = prover.ct_log2_size
    tr = api.Keccak256Transcript()

    def out_claims(t):
        p0 = t.squeeze_challenges(L)
        v0 = api.mle_eval_batch(ctx, d_ct[0], 1, L, p0)[0]
        p1 = t.squeeze_challenges(L)
        v1 = api.mle_eval_batch(ctx, d_ct[1], 1, L, p1)[0]
        return api._pk_output_claims(p0, v0, p1, v1)

    world, cap = 2, prover.circuit.shard_words
    gathered = torch.zeros(world * cap, dtype=torch.int64, device="cuda")
    merged = torch.zeros(cap, dtype=torch.int64, device="cuda")
    n = None
    for rank in (1, 0):                      # rank 0 last: its circuit keeps the deferred serialisers
        t = tr if rank == 0 else api.Keccak256Transcript()
        part = torch.zeros(cap, dtype=torch.int64, device="cuda")
        nw = prover.circuit.prove_gkr_shard_dev(out_claims(t), t, rank, world, part.data_ptr(), cap)
        ctx.synchronize()
        assert n is None or n == nw
        n = nw
        gathered[rank * n:(rank + 1) * n] = part[:n]
    torch.cuda.synchronize()
    api.shard_merge_device(ctx, gathered.data_ptr(), world, n, merged.data_ptr())
    claims = prover.circuit.emit_shard_dev(merged.data_ptr(), n)
    assert tr.into_proof() == want and same_claims(claims, wclaims)


@pytest.mark.gpu
def test_full_size_device_proof_equals_restatement(api, ctxs):
    """n = 32768, K = 16, Goldilocks: the first Lasso node of 22 variables (3 407 872 rows) on the device. A device witness is proved;
    bytes and input claims equal the restatement's on the downloaded witness; the host verifier and the batched verifier accept."""
    from hyper_greco_b200 import params, witness
    P = params.PK_PARAMS["32768_16x59_65537"]
    assert witness.pk_lasso_num_vars(P) == 22 and sum(l for _, l in witness.pk_lasso_lookup_segments(P)) == 3407872
    ctx = ctxs[0]
    dev, d_ct0, d_ct1 = witness.synth_pk_witness_device(ctx, P, 5)
    prover = api.BfvPkEncryptProver(ctx, P)
    proof, claims = prover.prove(dev, d_ct0, d_ct1)
    host, c0, c1 = device_limbs(ctx, dev, d_ct0, d_ct1, P)
    r = PkRestatement(0, P)
    r.evaluate(host)
    want, wclaims = r.prove(c0, c1)
    assert proof == want
    assert same_claims(claims, wclaims)
    v = api.BfvPkEncryptVerifier(P)
    v.verify(host, c0, c1, proof)
    for ins, t0, t1 in ((dev, d_ct0, d_ct1), (host, c0, c1)):   # a batch's tables are all on the device or all host vectors
        res = v.verify_batch(ctx, [ins, ins], [t0, t0], [t1, t1], [proof, proof[:-16]])
        assert [ok for ok, _ in res] == [True, False]
    prover.circuit.free()
    prover.lasso.free()


@pytest.mark.gpu
def test_bn254_8192_device_witness_proof_verifies(api, ctxs):
    from hyper_greco_b200 import params, witness
    P = params.PK_PARAMS["8192_4x55_65537"]
    ctx = ctxs[1]
    dev, d_ct0, d_ct1 = witness.synth_pk_witness_device(ctx, P, 6)
    prover = api.BfvPkEncryptProver(ctx, P)
    proof, claims = prover.prove(dev, d_ct0, d_ct1)
    host, c0, c1 = device_limbs(ctx, dev, d_ct0, d_ct1, P)
    v = api.BfvPkEncryptVerifier(P, api.BN254)
    assert same_claims(v.verify(host, c0, c1, proof), claims)
    assert [ok for ok, _ in v.verify_batch(ctx, [dev], [d_ct0], [d_ct1], [proof])] == [True]
    prover.circuit.free()
    prover.lasso.free()


def _host_verdict(api, v, ins, c0, c1, proof):
    try:
        v.verify(ins, c0, c1, proof)
        return True
    except api.HgError:
        return False


@pytest.mark.gpu
@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
def test_mixed_batches_get_the_host_verdicts(api, ctxs, field):
    """Shared points: every tamper case sits between good proofs. Per-proof points: absorbing caller transcripts, one proof flipped."""
    name = "1024_1x27_65537"
    P, _, flat, ct0, ct1 = instance(field, name)
    proof, _ = restatement_proof(field, name)
    v = api.BfvPkEncryptVerifier(P, field)
    ctx = ctxs[field]
    for label, ins, c0, c1, pr in tamper_cases(api, field, name):
        batch = [(flat, ct0, ct1, proof), (ins, c0, c1, pr), (flat, ct0, ct1, proof)]
        res = v.verify_batch(ctx, *[[b[k] for b in batch] for k in range(4)])
        assert [ok for ok, _ in res] == [_host_verdict(api, v, *b) for b in batch] == [True, False, True], label
    # per-proof points
    prover = api.BfvPkEncryptProver(ctx, P)
    items = []
    for seed in (1, 2):
        inner = Absorbing(field, seed)
        prover.prove_host(flat, ct0, ct1, api.MODE_INTERACTIVE, transcript=api.CallbackTranscript(inner, field))
        items.append((seed, inner.into_proof()))
    L = v.ct_log2_size

    def host(seed, pr):
        t = api.CallbackTranscript(Absorbing(field, seed, pr), field)
        p0, p1 = t.squeeze_challenges(L), t.squeeze_challenges(L)
        oc = api._pk_output_claims(p0, api.mle_eval_host(field, ct0, L, p0), p1, api.mle_eval_host(field, ct1, L, p1))
        try:
            return claims_match_inputs(api, field, flat, v.circuit.verify_gkr(oc, t))
        except api.HgError:
            return False

    for flip_seed in (None, 2):
        prs = []
        for seed, pr in items:
            if seed == flip_seed:
                pr = pr.copy()
                pr[len(pr) // 3] ^= 1
            prs.append((seed, pr))
        trs = [api.CallbackTranscript(Absorbing(field, s, pr), field) for s, pr in prs]
        got = [ok for ok, _ in v.verify_batch(ctx, [flat] * 2, [ct0] * 2, [ct1] * 2, trs)]
        assert got == [host(s, pr) for s, pr in prs] == [True, flip_seed is None]
    prover.circuit.free()
    prover.lasso.free()
