"""Vanilla layers with arbitrary multiplication gates (the two-phase layer sumcheck of DESIGN.md section 3, assumption A11).

Small circuits in both fields mix a general layer with linear, element-wise product, FFT and input nodes, and fan outputs out so that
nodes receive several claims. On the CPU: the CPU restatement (the oracle, with general layers restated in
tests/general_layer_oracle.cpp) proves and verifies them, every input claim equals the input's MLE, the library's host verifier
accepts the restatement's proofs with the same input claims, and changing any single proof element makes both verifiers reject.
On the GPU (-m gpu): the device evaluates and proves them with the restatement's values, bytes and claims in every schedule, and a
sharded proof gives the same bytes."""
import ctypes as C

import numpy as np
import pytest

GL_P = 2**64 - 2**32 + 1
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
PRIME = {0: GL_P, 1: BN_R}
FIELDS = [pytest.param(0, id="goldilocks"), pytest.param(1, id="bn254")]


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, build
    build.build()
    api.lib()
    return api


@pytest.fixture(scope="module")
def hgo():
    from oracle import hgo
    hgo.build()
    hgo.lib()
    return hgo


# ------------------------------------------------------------------------------------------------ CPU restatement of general layers
# tests/general_layer_oracle.cpp: the oracle (oracle/gkr.hpp) for every other node shape, an independent restatement of the
# two-phase layer sumcheck for general layers. Compiled with g++ into the temporary directory (the tree may be read-only),
# once per source version.
_GLIB = None


def _hgo():
    from oracle import hgo
    return hgo


def _glib():
    global _GLIB
    if _GLIB is None:
        import hashlib
        import os
        import subprocess
        import tempfile
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        src = os.path.join(root, "tests", "general_layer_oracle.cpp")
        deps = [src] + [os.path.join(root, "oracle", f) for f in sorted(os.listdir(os.path.join(root, "oracle"))) if f.endswith(".hpp")]
        tag = hashlib.sha256(b"".join(open(d, "rb").read() for d in deps)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"hg_general_layer_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.check_call([cxx, "-O3", "-march=x86-64-v3", "-std=c++17", "-fopenmp", "-fPIC", "-shared", "-w",
                                   "-I", os.path.join(root, "oracle"), "-o", tmp, src])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.hgt_last_error.restype = C.c_char_p
        _GLIB = L
    return _GLIB


def _gp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _gchk(rc):
    if rc != 0:
        raise _hgo().OracleError(_glib().hgt_last_error().decode())


def gates_to_csr(gates, field):
    """VanillaGate list -> the CSR arrays of hg_circuit_insert_vanilla. A gate is any object with `const` (None or int), `adds`
    [(coef, (input, wire))] and `muls` [(coef, (input, wire), (input, wire))]; a coefficient None is one."""
    one = lambda c: 1 if c is None else int(c)
    has_const = np.array([g.const is not None for g in gates], np.uint8)
    consts = _hgo().ints_to_limbs([0 if g.const is None else int(g.const) for g in gates], field)
    add_ptr, mul_ptr = np.zeros(len(gates) + 1, np.uint64), np.zeros(len(gates) + 1, np.uint64)
    ac, ai, aw, mc, m0, w0, m1, w1 = [], [], [], [], [], [], [], []
    for i, g in enumerate(gates):
        for c, (inp, w) in g.adds:
            ac.append(one(c)); ai.append(inp); aw.append(w)
        for c, (i0, x0), (i1, x1) in g.muls:
            mc.append(one(c)); m0.append(i0); w0.append(x0); m1.append(i1); w1.append(x1)
        add_ptr[i + 1], mul_ptr[i + 1] = len(ac), len(mc)
    u32 = lambda v: np.array(v, np.uint32)
    u64 = lambda v: np.array(v, np.uint64)
    return dict(has_const=has_const, consts=consts, add_ptr=add_ptr, add_coef=_hgo().ints_to_limbs(ac, field), add_in=u32(ai), add_wire=u64(aw),
                mul_ptr=mul_ptr, mul_coef=_hgo().ints_to_limbs(mc, field), mul_in0=u32(m0), mul_w0=u64(w0), mul_in1=u32(m1), mul_w1=u64(w1))


class GeneralOracle:
    """gkr::circuit::Circuit built node by node on the CPU restatement (the oracle plus tests/general_layer_oracle.cpp for general
    layers): insert / connect / evaluate / prove_gkr / verify_gkr. Points and values are limb arrays of extension elements ([nv, el]
    and [el]), as in the library's Circuit."""

    def __init__(self, field):
        L = _glib()
        vp, sz, i32p = C.c_void_p, C.c_size_t, C.POINTER(C.c_int)
        L.hgt_new.restype = vp
        L.hgt_new.argtypes = [C.c_int]
        L.hgt_free.argtypes = [vp]
        L.hgt_insert_input.argtypes = [vp, C.c_int, C.c_int, i32p]
        L.hgt_insert_fft.argtypes = [vp, C.c_int, C.c_int, i32p]
        L.hgt_insert_vanilla.argtypes = [vp, C.c_int, C.c_int, C.c_int, sz] + [vp] * 12 + [i32p]
        L.hgt_connect.argtypes = [vp, C.c_int, C.c_int]
        L.hgt_evaluate.argtypes = [vp, vp]
        L.hgt_value.argtypes = [vp, C.c_int, vp, C.POINTER(sz)]
        L.hgt_prove.argtypes = [vp, sz, vp, vp, vp, vp, sz, C.POINTER(sz)]
        L.hgt_verify.argtypes = [vp, sz, vp, vp, vp, vp, sz]
        L.hgt_num_inputs.restype = sz
        L.hgt_num_inputs.argtypes = [vp]
        L.hgt_num_claims.restype = sz
        L.hgt_num_claims.argtypes = [vp, sz]
        L.hgt_claim.argtypes = [vp, sz, sz, vp, vp, C.POINTER(sz)]
        self.field = field
        self.h = L.hgt_new(field)
        if not self.h:
            raise _hgo().OracleError(L.hgt_last_error().decode())

    def _id(self, fn, *args):
        i = C.c_int(-1)
        _gchk(fn(self.h, *args, C.byref(i)))
        return i.value

    def insert_input(self, log2_size, num_reps=1):
        return self._id(_glib().hgt_insert_input, log2_size, num_reps)

    def insert_fft(self, log2_size, inverse=False):
        return self._id(_glib().hgt_insert_fft, log2_size, 1 if inverse else 0)

    def insert_vanilla(self, arity, log2_sub, gates, num_reps=1):
        a = gates_to_csr(gates, self.field)
        keys = ("has_const", "consts", "add_ptr", "add_coef", "add_in", "add_wire", "mul_ptr", "mul_coef", "mul_in0", "mul_w0", "mul_in1", "mul_w1")
        return self._id(_glib().hgt_insert_vanilla, arity, log2_sub, num_reps, len(gates), *[_gp(np.ascontiguousarray(a[k])) for k in keys])

    def connect(self, frm, to):
        _gchk(_glib().hgt_connect(self.h, frm, to))

    def evaluate(self, inputs):
        """inputs: limb arrays of the input nodes, insertion order"""
        _gchk(_glib().hgt_evaluate(self.h, _gp(np.ascontiguousarray(np.concatenate([np.asarray(x, np.uint64).reshape(-1) for x in inputs]), np.uint64))))

    def value(self, node_id):
        n = C.c_size_t(0)
        _gchk(_glib().hgt_value(self.h, node_id, None, C.byref(n)))
        out = np.zeros(n.value * _hgo().LIMBS[self.field], np.uint64)
        _gchk(_glib().hgt_value(self.h, node_id, _gp(out), C.byref(n)))
        return out

    @staticmethod
    def _claims(output_claims):
        lens = np.array([len(p) for p, _ in output_claims], np.uint64)
        pts = np.concatenate([np.asarray(p, np.uint64).reshape(-1) for p, _ in output_claims] + [np.zeros(0, np.uint64)])
        vals = np.concatenate([np.asarray(v, np.uint64).reshape(-1) for _, v in output_claims] + [np.zeros(0, np.uint64)])
        return lens, np.ascontiguousarray(pts), np.ascontiguousarray(vals)

    def _input_claims(self):
        el = _hgo().LIMBS[self.field] * _hgo().DEGREE[self.field]
        out = []
        for i in range(_glib().hgt_num_inputs(self.h)):
            cl = []
            for k in range(_glib().hgt_num_claims(self.h, i)):
                nv = C.c_size_t(0)
                _gchk(_glib().hgt_claim(self.h, i, k, None, None, C.byref(nv)))
                pt, v = np.zeros((nv.value, el), np.uint64), np.zeros(el, np.uint64)
                _gchk(_glib().hgt_claim(self.h, i, k, _gp(pt), _gp(v), C.byref(nv)))
                cl.append((pt, v))
            out.append(cl)
        return out

    def prove_gkr(self, output_claims):
        """prove_gkr from a fresh transcript on the last evaluation -> (proof bytes, claims per input node [(point, value)])"""
        lens, pts, vals = self._claims(output_claims)
        n = C.c_size_t(0)
        buf = np.zeros(1 << 22, np.uint8)
        _gchk(_glib().hgt_prove(self.h, len(output_claims), _gp(lens), _gp(pts), _gp(vals), _gp(buf), buf.size, C.byref(n)))
        if n.value > buf.size:  # proved again into a buffer that fits
            buf = np.zeros(n.value, np.uint8)
            _gchk(_glib().hgt_prove(self.h, len(output_claims), _gp(lens), _gp(pts), _gp(vals), _gp(buf), buf.size, C.byref(n)))
        return buf[: n.value].tobytes(), self._input_claims()

    def verify_gkr(self, output_claims, proof: bytes):
        """verify_gkr on a fresh transcript holding `proof`; raises OracleError on rejection; returns the input claims"""
        lens, pts, vals = self._claims(output_claims)
        buf = np.frombuffer(proof, np.uint8).copy() if proof else np.zeros(0, np.uint8)
        _gchk(_glib().hgt_verify(self.h, len(output_claims), _gp(lens), _gp(pts), _gp(vals), _gp(buf), buf.size))
        return self._input_claims()

    def __del__(self):
        try:
            _glib().hgt_free(self.h)
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------ circuits
# A circuit is a list of ops applied in order to any builder with insert_input / insert_fft / insert_vanilla / connect:
# ("input", log2_size, num_reps), ("fft", log2_size, inverse), ("vanilla", arity, log2_sub, gates, num_reps), ("connect", from, to).
def _gate(api, const=None, adds=(), muls=()):
    return api.VanillaGate(const=const, adds=list(adds), muls=list(muls))


def circuit_mixed(api, p):
    """A general layer of arity 3 (a_pad 4) with 5 gates next to every other node shape; `em` and `a` fan out."""
    G = lambda **k: _gate(api, **k)
    ops = [("input", 3, 1), ("input", 3, 1), ("input", 2, 2)]                       # 0 a, 1 b, 2 c (num_reps 2: 8 elements)
    ops += [("fft", 3, False)]                                                       # 3 f = FFT(a)
    ops += [("vanilla", 2, 3, [G(adds=[(None, (0, i)), (3, (1, 7 - i))]) for i in range(8)], 1)]          # 4 lin = a + 3 b~
    ops += [("vanilla", 2, 3, [G(muls=[(None, (0, i), (1, i))]) for i in range(8)], 1)]                   # 5 em = f * b
    gen = [G(const=5, muls=[(None, (0, 0), (1, 1))]),                                # constant + product of two different wires
           G(adds=[(None, (1, 3))], muls=[(p - 1, (0, 2), (0, 2))]),                 # (p - 1) * square + add
           G(adds=[(2, (0, 5))], muls=[(0, (2, 4), (1, 6)), (None, (2, 1), (0, 7))]),  # coefficient 0, a product, an add
           G(const=0, muls=[(None, (1, 0), (2, 0)), (None, (0, 1), (1, 1))]),
           G(muls=[(7, (2, 7), (2, 7))])]
    ops += [("vanilla", 3, 3, gen, 1)]                                               # 6 gen(lin, em, c)
    ops += [("vanilla", 1, 3, [G(adds=[(None, (0, i))]) for i in range(8)], 1)]      # 7 relay of em: em gets two claims
    reps = [G(muls=[(None, (0, 1), (1, 2))]), G(const=7, muls=[(None, (0, 3), (0, 3))], adds=[(p - 1, (1, 0))]), G(muls=[(4, (1, 3), (0, 0))])]
    ops += [("vanilla", 2, 2, reps, 2)]                                              # 8 general, num_reps 2, 3 gates per rep, over (c, lin)
    ops += [("connect", 0, 3), ("connect", 0, 4), ("connect", 1, 4), ("connect", 3, 5), ("connect", 1, 5),
            ("connect", 4, 6), ("connect", 5, 6), ("connect", 2, 6), ("connect", 5, 7), ("connect", 2, 8), ("connect", 4, 8)]
    return ops


def circuit_square(api, p):
    """out[i] = in[i]^2 (in0 == in1, w0 == w1) of one input, arity 1, and a fan-out of its input into a linear layer"""
    G = lambda **k: _gate(api, **k)
    return [("input", 4, 1), ("vanilla", 1, 4, [G(muls=[(None, (0, i), (0, i))]) for i in range(16)], 1),
            ("vanilla", 1, 4, [G(adds=[(None, (0, 15 - i))]) for i in range(16)], 1), ("connect", 0, 1), ("connect", 0, 2)]


def circuit_one_gate(api, p):
    """a layer of one gate: 2 + (p - 1) a[3] b[5] + a[0]"""
    G = lambda **k: _gate(api, **k)
    return [("input", 3, 1), ("input", 3, 1), ("vanilla", 2, 3, [G(const=2, adds=[(None, (0, 0))], muls=[(p - 1, (0, 3), (1, 5))])], 1),
            ("connect", 0, 2), ("connect", 1, 2)]


def circuit_random(api, p, seed=11):
    """random wiring: arity 3, num_reps 2, 11 gates per rep, each with up to 3 products and 2 adds and an optional constant"""
    rng = np.random.default_rng(seed)
    G = lambda **k: _gate(api, **k)
    sub, ar = 8, 3
    wire = lambda: (int(rng.integers(0, ar)), int(rng.integers(0, sub)))
    coef = lambda: [None, 0, 1, p - 1, int(rng.integers(0, 2**62))][int(rng.integers(0, 5))]
    gates = [G(const=None if rng.random() < 0.5 else int(rng.integers(0, 2**62)),
               adds=[(coef(), wire()) for _ in range(int(rng.integers(0, 3)))],
               muls=[(coef(), wire(), wire()) for _ in range(int(rng.integers(1, 4)))]) for _ in range(11)]
    ops = [("input", 4, 1), ("input", 3, 2), ("input", 4, 1), ("vanilla", ar, 3, gates, 2)]
    return ops + [("connect", 0, 3), ("connect", 1, 3), ("connect", 2, 3)]


CASES = {"mixed": circuit_mixed, "square": circuit_square, "one_gate": circuit_one_gate, "random": circuit_random}


def build(builder, ops):
    ids = []
    for op in ops:
        if op[0] == "input":
            ids.append(builder.insert_input(op[1], op[2]))
        elif op[0] == "fft":
            ids.append(builder.insert_fft(op[1], op[2]))
        elif op[0] == "vanilla":
            ids.append(builder.insert_vanilla(op[1], op[2], op[3], op[4]))
        else:
            builder.connect(op[1], op[2])
    return ids


def node_shapes(ops):
    """(kind, out_len) per node, and the output nodes (no successors, not inputs) in insertion order"""
    nodes, succ = [], []
    for op in ops:
        if op[0] == "input":
            nodes.append(("input", op[2] << op[1]))
        elif op[0] == "fft":
            nodes.append(("fft", 1 << op[1]))
        elif op[0] == "vanilla":
            n = len(op[3]) * op[4]
            nodes.append(("vanilla", 1 << (n - 1).bit_length()))
        else:
            succ.append(op[1])
    outs = [i for i, (k, _) in enumerate(nodes) if k != "input" and i not in succ]
    return nodes, outs


def rand_ext(field, rng, n):
    """n random extension elements as limbs [n, el]"""
    from oracle import hgo
    if field == 0:
        return rng.integers(0, GL_P, size=(n, 2), dtype=np.uint64)
    vals = [int(rng.integers(0, 2**63)) * 2**190 % BN_R + int(rng.integers(0, 2**63)) for _ in range(n)]
    return hgo.ints_to_limbs(vals, 1).reshape(n, 4)


def make_instance(hgo, api, field, case, seed=0):
    """-> (ops, oracle circuit, input limb arrays, output claims) with the oracle evaluated on random inputs"""
    rng = np.random.default_rng(seed)
    ops = CASES[case](api, PRIME[field])
    nodes, outs = node_shapes(ops)
    oc = GeneralOracle(field)
    build(oc, ops)
    ins = []
    for kind, n in nodes:
        if kind == "input":
            ins.append(hgo.ints_to_limbs([int(rng.integers(0, 2**62)) * (1 + int(rng.integers(0, 2**60))) % PRIME[field] for _ in range(n)], field))
    oc.evaluate(ins)
    claims = []
    for o in outs:
        nv = (nodes[o][1] - 1).bit_length()
        pt = rand_ext(field, rng, nv)
        claims.append((pt, hgo.mle_eval(field, oc.value(o), nv, pt)))
    return ops, oc, ins, claims


def same_claims(a, b):
    return len(a) == len(b) and all(len(x) == len(y) and all((p.reshape(-1) == q.reshape(-1)).all() and (v == w).all() for (p, v), (q, w) in zip(x, y))
                                    for x, y in zip(a, b))


def host_verify(api, ops, field, claims, proof):
    c = api.Circuit(None, field)
    build(c, ops)
    return c.verify_gkr(claims, api.Keccak256Transcript.from_proof(proof, field))


def element_flips(proof, field):
    """every proof element, one at a time, replaced by itself + 1 (still canonical)"""
    bsz = 8 * (1 if field == 0 else 4)
    esz = bsz * (2 if field == 0 else 1)
    assert len(proof) % esz == 0
    for off in range(0, len(proof), esz):
        v = (int.from_bytes(proof[off:off + bsz], "big") + 1) % PRIME[field]
        yield proof[:off] + v.to_bytes(bsz, "big") + proof[off + bsz:]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("field", FIELDS)
def test_oracle_prove_verify_and_host_verifier(api, hgo, field, case):
    ops, oc, ins, claims = make_instance(hgo, api, field, case)
    proof, pclaims = oc.prove_gkr(claims)
    vclaims = oc.verify_gkr(claims, proof)
    assert same_claims(pclaims, vclaims)
    for vec, cl in zip(ins, pclaims):
        assert cl
        for pt, v in cl:
            assert (hgo.mle_eval(field, vec, pt.shape[0], pt) == v).all()
    assert same_claims(host_verify(api, ops, field, claims, proof), pclaims)


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("field", FIELDS)
def test_every_flipped_element_is_rejected(api, hgo, field, case):
    ops, oc, ins, claims = make_instance(hgo, api, field, case)
    proof, _ = oc.prove_gkr(claims)
    n = 0
    for bad in element_flips(proof, field):
        with pytest.raises(hgo.OracleError):
            oc.verify_gkr(claims, bad)
        with pytest.raises(api.HgError):
            host_verify(api, ops, field, claims, bad)
        n += 1
    assert n > 10


def test_general_layer_classification_in_the_oracle(api, hgo):
    """the element-wise product path is taken only for out[i] = in0[i] * in1[i] with num_reps 1: with num_reps 2 the same gates
    form a general layer (and the proof has two sumchecks, so it is longer than an element-wise one would be)"""
    G = lambda **k: _gate(api, **k)
    ew = [G(muls=[(None, (0, i), (1, i))]) for i in range(4)]
    for reps in (1, 2):
        oc = GeneralOracle(0)
        build(oc, [("input", 2, reps), ("input", 2, reps), ("vanilla", 2, 2, ew, reps), ("connect", 0, 2), ("connect", 1, 2)])
        rng = np.random.default_rng(reps)
        ins = [rng.integers(0, GL_P, size=4 * reps, dtype=np.uint64) for _ in range(2)]
        oc.evaluate(ins)
        nv = (4 * reps - 1).bit_length()
        pt = rand_ext(0, rng, nv)
        proof, _ = oc.prove_gkr([(pt, hgo.mle_eval(0, oc.value(2), nv, pt))])
        elems = len(proof) // 16
        if reps == 1:
            assert elems == nv * 3 + 2            # degree-3 rounds (3 elements each) + two input evaluations
        else:
            assert elems == 2 * (4 * 2) + 2 * 2  # two phases of nv = 4 degree-2 rounds + two evaluations after each


@pytest.mark.parametrize("which", ["has_const", "consts"])
def test_insert_vanilla_rejects_null_arrays(api, which):
    """hg_circuit_insert_vanilla checks its pointers before it copies anything"""
    c = api.Circuit(None, api.GOLDILOCKS)
    c.insert_input(1, 1)
    one = np.ones(1, np.uint8)
    z = np.zeros(2, np.uint64)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    args = {"has_const": ptr(one), "consts": ptr(z)}
    args[which] = None
    i = C.c_int(-1)
    rc = api.lib().hg_circuit_insert_vanilla(c.h, 1, 1, 1, 1, args["has_const"], args["consts"], ptr(z), None, None, None, ptr(z), None, None, None,
                                             None, None, C.byref(i))
    assert rc != 0 and i.value == -1
    # the same call with both arrays inserts a constant gate
    rc = api.lib().hg_circuit_insert_vanilla(c.h, 1, 1, 1, 1, ptr(one), ptr(z), ptr(z), None, None, None, ptr(z), None, None, None, None, None, C.byref(i))
    assert rc == 0 and i.value == 1


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctxs(api):
    made = {}

    def get(field):
        if field not in made:
            made[field] = api.Context(0, field)
        return made[field]
    yield get
    for c in made.values():
        c.close()


def device_circuit(api, ctx, ops, ins):
    c = api.Circuit(ctx)
    ids = build(c, ops)
    c.evaluate_host(ins)
    return c, ids


def device_values(api, ctx, c, node_id):
    ptr, n = c.node_value(node_id)
    k = api.LIMBS[ctx.field]
    raw = api.NodeValueView(ctx, ptr, n).download(np.uint64, n * k)
    if k == 1:
        return raw
    tmp = api.DeviceBuffer(ctx, raw.nbytes)
    tmp.upload(raw)
    return tmp.to_field(n).reshape(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("field", FIELDS)
def test_device_matches_oracle(api, hgo, ctxs, field, case):
    """device evaluate == oracle evaluate; proof bytes and input claims == the oracle's in prefetch and interactive mode and with a
    callback transcript"""
    ctx = ctxs(field)
    ops, oc, ins, claims = make_instance(hgo, api, field, case)
    want, wclaims = oc.prove_gkr(claims)
    c, ids = device_circuit(api, ctx, ops, ins)
    for i in ids:
        assert (device_values(api, ctx, c, i) == oc.value(i)).all(), i
    for mode in (api.MODE_PREFETCH, api.MODE_INTERACTIVE):
        tr = api.Keccak256Transcript(field)
        got = c.prove_gkr(claims, tr, mode)
        assert tr.into_proof() == want, mode
        assert same_claims(got, wclaims), mode
    tr = api.CallbackTranscript(api.Keccak256Transcript(field), field)
    got = c.prove_gkr(claims, tr, api.MODE_PREFETCH)
    assert tr.into_proof() == want and same_claims(got, wclaims)
    c.free()


def _emulate_ranks(api, ctx, world, cap_words, prove_shard_dev, emit):
    """every rank of one sharded proof emulated on this device: partial buffers gathered, merged by one kernel, emitted"""
    import torch
    gathered = torch.zeros(world * cap_words, dtype=torch.int64, device="cuda")
    merged = torch.zeros(cap_words, dtype=torch.int64, device="cuda")
    n = None
    for r in range(world - 1, -1, -1):  # rank 0 last: its circuit keeps the serialisers
        part = torch.zeros(cap_words, dtype=torch.int64, device="cuda")
        nw = prove_shard_dev(r, world, part.data_ptr(), cap_words)
        ctx.synchronize()
        assert n is None or n == nw
        n = nw
        gathered[r * n:(r + 1) * n] = part[:n]
    torch.cuda.synchronize()
    api.shard_merge_device(ctx, gathered.data_ptr(), world, n, merged.data_ptr())
    return emit(merged.data_ptr(), n)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("field", FIELDS)
def test_sharded_equals_single_device(api, hgo, ctxs, field, world):
    ctx = ctxs(field)
    ops, oc, ins, claims = make_instance(hgo, api, field, "mixed")
    c, _ = device_circuit(api, ctx, ops, ins)
    tr0 = api.Keccak256Transcript(field)
    claims0 = c.prove_gkr(claims, tr0, api.MODE_PREFETCH)
    want = tr0.into_proof()
    tr = api.Keccak256Transcript(field)
    shard = lambda r, w, ptr, cap: c.prove_gkr_shard_dev(claims, tr if r == 0 else api.Keccak256Transcript(field), r, w, ptr, cap)
    got = _emulate_ranks(api, ctx, world, c.shard_words, shard, c.emit_shard_dev)
    assert tr.into_proof() == want and same_claims(got, claims0)
    # the per-rank parts of the serialisation concatenate to the same proof
    tr = api.Keccak256Transcript(field)
    parts = []

    def emit_parts(d_merged, n):
        for p in range(world):
            parts.append(c.emit_shard_part_dev(d_merged, n, p, world))
            assert same_claims(c._read_input_claims(), claims0)
    _emulate_ranks(api, ctx, world, c.shard_words, shard, emit_parts)
    for x in parts:
        tr.append_bytes(x)
    assert tr.into_proof() == want
    c.free()


@pytest.mark.gpu
def test_large_general_layer_verifies(api, hgo, ctxs):
    """one general layer of S = 2^20 (arity 2, num_reps 16, 2^15 gates per rep, random wiring) on the device: the host verifier
    accepts the proof and every input claim equals the input's MLE"""
    ctx = ctxs(0)
    rng = np.random.default_rng(5)
    log2_sub, reps, ng = 15, 16, 1 << 15
    sub = 1 << log2_sub
    n_in = reps * sub
    w = lambda k: rng.integers(0, sub, size=k)
    i0, i1, x0, x1 = rng.integers(0, 2, size=ng), rng.integers(0, 2, size=ng), w(ng), w(ng)
    coef = rng.integers(0, GL_P, size=ng, dtype=np.uint64)
    has_const = rng.random(ng) < 0.25
    consts = rng.integers(0, GL_P, size=ng, dtype=np.uint64)
    add_ptr = np.arange(ng + 1, dtype=np.uint64)
    mul_ptr = np.arange(ng + 1, dtype=np.uint64)
    arrays = (2, log2_sub, reps, has_const.astype(np.uint8), consts, add_ptr, rng.integers(0, GL_P, size=ng, dtype=np.uint64),
              rng.integers(0, 2, size=ng).astype(np.uint32), w(ng).astype(np.uint64), mul_ptr, coef, i0.astype(np.uint32), x0.astype(np.uint64),
              i1.astype(np.uint32), x1.astype(np.uint64))
    ins = [rng.integers(0, GL_P, size=n_in, dtype=np.uint64) for _ in range(2)]
    c = api.Circuit(ctx)
    a, b = c.insert_input(log2_sub, reps), c.insert_input(log2_sub, reps)
    g = c.insert_vanilla_arrays(*arrays)
    c.connect(a, g)
    c.connect(b, g)
    c.evaluate_host(ins)
    nv = (ng * reps - 1).bit_length()
    pt = rand_ext(0, rng, nv)
    ptr, n = c.node_value(g)
    out = api.NodeValueView(ctx, ptr, n).download(np.uint64, n)
    claims = [(pt, hgo.mle_eval(0, out, nv, pt))]
    tr = api.Keccak256Transcript()
    got = c.prove_gkr(claims, tr, api.MODE_PREFETCH)
    proof = tr.into_proof()
    h = api.Circuit(None, api.GOLDILOCKS)
    ha, hb = h.insert_input(log2_sub, reps), h.insert_input(log2_sub, reps)
    hg = h.insert_vanilla_arrays(*arrays)
    h.connect(ha, hg)
    h.connect(hb, hg)
    vclaims = h.verify_gkr(claims, api.Keccak256Transcript.from_proof(proof))
    assert same_claims(got, vclaims)
    for vec, cl in zip(ins, vclaims):
        assert len(cl) == 2
        for p, v in cl:
            assert (hgo.mle_eval(0, vec, p.shape[0], p) == v).all()
    c.free()
