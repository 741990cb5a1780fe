"""Batched verification of BfvEncrypt proofs on the device (hg_verifier_new / hg_gkr_verify_batch / hg_mle_eval_multi,
api.BfvSkEncryptVerifier.verify_batch). Every verdict is compared with the host verifier (hg_gkr_verify + hg_mle_eval_host, i.e.
BfvSkEncryptVerifier.verify), proof by proof."""
import gc
import hashlib
import os

import numpy as np
import pytest

GL_P = 2**64 - 2**32 + 1
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, build
    build.build()
    api.lib()
    return api


def golden_io(field):
    name = "1024_1x27_65537"
    io = np.load(os.path.join(GOLDEN, ("circuit_io_{}.npz" if field == 0 else "circuit_io_bn254_{}.npz").format(name)))
    flat = [np.ascontiguousarray(v, np.uint64).reshape(-1) for v in [io["s"], io["e"], io["k1"]] + list(io["ais"]) + list(io["r1is"]) + [io["r2is"]]]
    ct = np.ascontiguousarray(io["ct0is"], np.uint64).reshape(-1)
    tag = "goldilocks" if field == 0 else "bn254"
    proof = open(os.path.join(GOLDEN, f"proof_{tag}_bfv_encrypt_{name}.bin"), "rb").read()
    return name, flat, ct, proof


def host_verdict(api, v, flat, ct, proof, options=None):
    try:
        v.verify(flat, ct, proof, options)
        return True
    except api.HgError:
        return False


def flat_inputs(ins):
    return [np.array(v, dtype=np.uint64).reshape(-1) for v in [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]]


# ------------------------------------------------------------------------------------------------------------------------ CPU
def test_compute_calls_fail_without_a_gpu(api):
    """The new entry points are callable from the library and refuse NULL handles with an error, never a crash; without a device no
    context can be made, and every compute call of the batch verifier needs one."""
    import ctypes as C
    L = api.lib()
    assert L.hg_gkr_verify_batch(None, 0, None, 0, None, None, None, None, 0, None, None) != 0
    assert L.hg_mle_eval_multi(None, 0, None, None, None, 0, None) != 0
    assert L.hg_verifier_new(None, None, 1, C.byref(C.c_void_p())) != 0
    assert L.hg_verifier_reason(None, 0) == b""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if not has_gpu:
        with pytest.raises(api.HgError):
            api.Context(0)


# ------------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctxs(api):
    c = {0: api.Context(0, api.GOLDILOCKS), 1: api.Context(0, api.BN254)}
    yield c
    gc.collect()  # the tests' provers and verifiers go before the contexts they were made on
    for x in c.values():
        x.close()


@pytest.mark.gpu
@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
def test_golden_proofs_and_tampering_in_mixed_batches(api, ctxs, field):
    """The golden proofs are accepted in a batch; each tamper case of the host verifier's test sits in a batch between good proofs,
    and exactly that proof is rejected, with the host verifier's verdict; a flip inside the Lasso node's discarded sumcheck
    outputs is accepted, as the reference does; host vectors and device tables give the same verdicts."""
    from hyper_greco_b200 import params
    name, flat, ct, proof = golden_io(field)
    P = params.PARAMS[name]
    v = api.BfvSkEncryptVerifier(P, field)
    ctx = ctxs[field]
    step = 16 if field == 0 else 32
    cases = []
    for off in (3, 5 * step + 1, len(proof) - 2, len(proof) - 40 * step):
        bad = bytearray(proof)
        bad[off] ^= 0x10
        cases.append((flat, ct, bytes(bad)))
    cases.append((flat, ct, proof[:-step]))
    cases.append((flat, ct, proof + proof[-step:]))
    ct_bad = ct.copy()
    ct_bad[0] ^= 1
    cases.append((flat, ct_bad, proof))
    s_bad = [x.copy() for x in flat]
    s_bad[0][0] ^= 1
    cases.append((s_bad, ct, proof))
    # element 205 lies in the Lasso node's grand-product sumcheck messages, whose final claims the reference discards
    # (verifier.rs:218-221): the host verifier accepts the flip, and so must the batch
    lasso = bytearray(proof)
    lasso[205 * step] ^= 0x01
    assert host_verdict(api, v, flat, ct, bytes(lasso))
    cases.append((flat, ct, bytes(lasso)))
    for fl, c, pr in cases:
        batch = [(flat, ct, proof), (fl, c, pr), (flat, ct, proof)]
        res = v.verify_batch(ctx, [b[0] for b in batch], [b[1] for b in batch], [b[2] for b in batch])
        want = [host_verdict(api, v, *b) for b in batch]
        assert [ok for ok, _ in res] == want
        assert res[0][0] and res[2][0] and res[0][1] == ""
        assert res[1][1] == "" if res[1][0] else res[1][1] != ""
    assert [host_verdict(api, v, *c) for c in cases] == [False] * (len(cases) - 1) + [True]
    # device-resident inputs: the library's representation
    d_in = [api.DeviceBuffer.from_numpy(ctx, x) for x in flat]
    d_ct = api.DeviceBuffer.from_numpy(ctx, ct)
    if field == 1:
        for b, x in zip(d_in + [d_ct], flat + [ct]):
            api._chk(api.lib().hg_field_encode(ctx.h, b.ptr, x.size // 4))
    res = v.verify_batch(ctx, [d_in, d_in], [d_ct, d_ct], [proof, proof[:-step]])
    assert [ok for ok, _ in res] == [True, False]


@pytest.mark.gpu
@pytest.mark.parametrize("n,seeds", [(4096, (1, 2, 3)), (32768, (5, 6))])
def test_device_proofs_match_the_host_verifier(api, ctxs, n, seeds):
    """Batches of device-made proofs of synthetic witnesses, each also paired with an altered input and a wrong ct0is: the verdict
    of every proof equals the host verifier's."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(n)
    ctx = ctxs[0]
    prover = api.BfvSkEncryptProver(ctx, P)
    v = api.BfvSkEncryptVerifier(P)
    batch = []
    for seed in seeds:
        ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, seed))
        flat = flat_inputs(ins)
        ct = np.array(ct0is, dtype=np.uint64)
        proof, _ = prover.prove_host(flat, ct, 0)
        batch.append((flat, ct, proof))
        alt = [x.copy() for x in flat]
        alt[3][7] = (int(alt[3][7]) + 1) % GL_P
        batch.append((alt, ct, proof))
        ct2 = ct.copy()
        ct2[-1] = (int(ct2[-1]) + 1) % GL_P
        batch.append((flat, ct2, proof))
    res = v.verify_batch(ctx, [b[0] for b in batch], [b[1] for b in batch], [b[2] for b in batch])
    want = [host_verdict(api, v, *b) for b in batch]
    assert [ok for ok, _ in res] == want
    assert want == [True, False, False] * len(seeds)


@pytest.mark.gpu
@pytest.mark.parametrize("a3w,a3h,a5", [(1, 0, 1), (0, 1, 0), (1, 1, 0)])
def test_non_default_switches(api, ctxs, a3w, a3h, a5):
    """Proofs made under non-default A3 / A3' / A5 settings verify with the matching options3, as on the host."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(4096)
    ctx = api.Context(0, api.GOLDILOCKS)
    ctx.set_option(api.OPT_A3_WIRE, a3w)
    ctx.set_option(api.OPT_A3_H1, a3h)
    ctx.set_option(api.OPT_A5_ASCENDING, a5)
    prover = api.BfvSkEncryptProver(ctx, P)
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, 9))
    flat, ct = flat_inputs(ins), np.array(ct0is, dtype=np.uint64)
    proof, _ = prover.prove_host(flat, ct, 0)
    v = api.BfvSkEncryptVerifier(P)
    opts = [a3w, a3h, a5]
    bad = bytearray(proof)
    bad[100] ^= 4
    batch = [proof, bytes(bad)]
    res = v.verify_batch(ctx, [flat] * 2, [ct] * 2, batch, opts)
    assert [ok for ok, _ in res] == [host_verdict(api, v, flat, ct, p, opts) for p in batch] == [True, False]
    # objects before their context: their destructors select the context's device
    v._batch.free()
    prover.circuit.free()
    prover.lasso.free()
    ctx.close()


class Absorbing:
    """A transcript whose squeeze hashes everything written or read so far: every proof gets its own points."""

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


@pytest.mark.gpu
def test_points_that_differ_per_proof(api, ctxs):
    """With an absorbing caller transcript every proof has its own points; the verdicts still equal the host verifier's."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(4096)
    ctx = ctxs[0]
    prover = api.BfvSkEncryptProver(ctx, P)
    v = api.BfvSkEncryptVerifier(P)
    L = prover.ct0is_log2_size
    items = []
    for seed in (1, 2):
        ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, seed))
        flat, ct = flat_inputs(ins), np.array(ct0is, dtype=np.uint64)
        inner = Absorbing(0, seed)
        tr = api.CallbackTranscript(inner, api.GOLDILOCKS)
        prover.circuit.evaluate_host(flat)
        d_ct = api.DeviceBuffer.from_numpy(ctx, ct)
        point = tr.squeeze_challenges(L)
        value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
        prover.circuit.prove_gkr([(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (point, value)], tr, api.MODE_INTERACTIVE)
        items.append((seed, flat, ct, inner.into_proof()))

    def run(mutate):
        trs, ins_l, cts, host = [], [], [], []
        for seed, flat, ct, pr in items:
            pr = mutate(seed, pr)
            trs.append(api.CallbackTranscript(Absorbing(0, seed, pr), api.GOLDILOCKS))
            ins_l.append(flat)
            cts.append(ct)
            # host verdict with the same transcript kind
            htr = api.CallbackTranscript(Absorbing(0, seed, pr), api.GOLDILOCKS)
            pt = htr.squeeze_challenges(L)
            val = api.mle_eval_host(0, ct, L, pt)
            try:
                claims = v.circuit.verify_gkr([(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (pt, val)], htr)
                host.append(all((api.mle_eval_host(0, vec, p.shape[0], p) == x).all() for vec, cl in zip(flat, claims) for p, x in cl))
            except api.HgError:
                host.append(False)
        res = v.verify_batch(ctx, ins_l, cts, trs)
        return [ok for ok, _ in res], host

    got, host = run(lambda s, p: p)
    assert got == host == [True, True]

    def flip(s, p):
        if s != 2:
            return p
        q = p.copy()
        q[len(q) // 3] = (int(q[len(q) // 3]) + 1) % GL_P
        return q
    got, host = run(flip)
    assert got == host and got[0] and not got[1]


@pytest.mark.gpu
def test_batch_limits(api, ctxs):
    """B = 1, 2 and max_batch work; max_batch + 1 is a call error, not a rejection."""
    from hyper_greco_b200 import params
    name, flat, ct, proof = golden_io(0)
    P = params.PARAMS[name]
    v = api.BfvSkEncryptVerifier(P, 0)
    ctx = ctxs[0]
    bv = api.GkrBatchVerifier(ctx, v.circuit, 3)
    L = v.ct0is_log2_size

    def run(k):
        trs = [api.Keccak256Transcript.from_proof(proof, 0) for _ in range(k)]
        pts = [t.squeeze_challenges(L) for t in trs]
        vals = api.mle_eval_multi(ctx, [ct] * k, pts)
        oc = [[(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (pts[i], vals[i])] for i in range(k)]
        return bv.verify_batch(trs, oc, [flat] * k)
    for k in (1, 2, 3):
        assert all(ok for ok, _ in run(k))
    with pytest.raises(api.HgError):
        run(4)
    bv.free()


@pytest.mark.gpu
@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
def test_mle_eval_multi_matches_the_host(api, ctxs, field):
    """Per-item MLEs of host and device tables at their own points equal hg_mle_eval_host."""
    rng = np.random.default_rng(3)
    ctx = ctxs[field]
    limbs, el = (1, 2) if field == 0 else (4, 4)
    p = GL_P if field == 0 else BN_R
    tabs, pts = [], []
    for nv in (0, 1, 5, 11, 13, 17):
        t = np.array([[int(x) % p >> (64 * j) & 0xFFFFFFFFFFFFFFFF for j in range(limbs)] for x in rng.integers(0, 2**62, 1 << nv)], np.uint64).reshape(-1)
        pt = np.array([[int(x) % p >> (64 * j) & 0xFFFFFFFFFFFFFFFF for j in range(el)] for x in rng.integers(0, 2**62, nv)], np.uint64).reshape(nv, el)
        tabs.append(t)
        pts.append(pt)
    got = api.mle_eval_multi(ctx, tabs, pts)
    for t, pt, g in zip(tabs, pts, got):
        assert (g == api.mle_eval_host(field, t, pt.shape[0], pt)).all()


def _general_layer_module():
    import importlib.util
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_general_layer.py")
    spec = importlib.util.spec_from_file_location("_general_layer_cases", path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["mixed", "square", "one_gate", "random"])
@pytest.mark.parametrize("field", [0, 1], ids=["goldilocks", "bn254"])
def test_general_layer_circuits_in_a_batch(api, ctxs, oracle, field, case):
    """The small circuits of test_general_layer.py (general layers next to linear, FFT and product layers, fan-out) proved by the
    CPU restatement: a batch of the proof, a proof with one element changed and the proof with a changed input gets the host
    verifier's verdicts (hg_gkr_verify followed by the input-claim check)."""
    gl = _general_layer_module()
    ops, oc, ins, claims = gl.make_instance(oracle, api, field, case)
    proof, _ = oc.prove_gkr(claims)
    bad = next(gl.element_flips(proof, field))
    ins_bad = [x.copy() for x in ins]
    ins_bad[0][0] = (int(ins_bad[0][0]) + 1) % gl.PRIME[field] if field == 0 else ins_bad[0][0] ^ 1
    desc = api.Circuit(None, field)
    gl.build(desc, ops)
    bv = api.GkrBatchVerifier(ctxs[field], desc, 3)

    def host(pr, inputs):
        try:
            cl = gl.host_verify(api, ops, field, claims, pr)
        except api.HgError:
            return False
        return all((api.mle_eval_host(field, vec, p.shape[0], p) == x).all() for vec, c in zip(inputs, cl) for p, x in c)
    batch = [(proof, ins), (bad, ins), (proof, ins_bad)]
    res = bv.verify_batch([api.Keccak256Transcript.from_proof(p, field) for p, _ in batch], [claims] * 3, [i for _, i in batch])
    assert [ok for ok, _ in res] == [host(p, i) for p, i in batch] == [True, False, False]
    bv.free()
