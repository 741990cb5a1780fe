"""Batched device verification of circuits with general Vanilla layers (hg_verifier_new / hg_gkr_verify_batch, api.GkrBatchVerifier).

The replay of a batch leaves a general layer's final check to the device: A(u), the constant part and M(u, v) are computed there,
once per batch for proofs that share their points. Every verdict here is compared with the host verifier's (hg_gkr_verify followed
by the input-claim check), proof by proof. The host verifier itself, which keeps checking general layers in full, is covered by
test_general_layer.py::test_oracle_prove_verify_and_host_verifier (its input claims equal the CPU restatement's) and
::test_every_flipped_element_is_rejected."""
import gc
import importlib.util
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = [pytest.param(0, id="goldilocks"), pytest.param(1, id="bn254")]
MAX_BATCH = 16


def _load(name):
    spec = importlib.util.spec_from_file_location("_gv_" + name, os.path.join(HERE, name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def circuit_kinds(api, p):
    """every kind the device verifier defers in one circuit: a general layer with constants and num_reps 2 over an element-wise
    product (of an FFT and an input) and a linear layer; two linear relays of the general layer make it take two claims (alpha)"""
    G = lambda **k: api.VanillaGate(const=k.get("const"), adds=list(k.get("adds", ())), muls=list(k.get("muls", ())))
    ops = [("input", 3, 1), ("input", 3, 1)]                                                      # 0 a, 1 b
    ops += [("fft", 3, False)]                                                                    # 2 f = FFT(a)
    ops += [("vanilla", 2, 3, [G(muls=[(None, (0, i), (1, i))]) for i in range(8)], 1)]          # 3 em = f * b
    ops += [("vanilla", 2, 3, [G(adds=[(None, (0, i)), (2, (1, 7 - i))]) for i in range(8)], 1)]  # 4 lin = a + 2 b~
    gen = [G(const=5, muls=[(None, (0, 1), (1, 2))]),
           G(adds=[(3, (1, 0))], muls=[(p - 1, (0, 3), (0, 3))]),
           G(const=9, adds=[(None, (0, 2))], muls=[(4, (1, 3), (0, 0)), (None, (1, 1), (1, 1))]),
           G(muls=[(7, (0, 2), (1, 3))])]
    ops += [("vanilla", 2, 2, gen, 2)]                                                            # 5 general(em, lin), 8 outputs
    ops += [("vanilla", 1, 3, [G(adds=[(None, (0, i))]) for i in range(8)], 1)]                  # 6 relay of the general layer
    ops += [("vanilla", 1, 3, [G(const=1, adds=[(3, (0, 7 - i))]) for i in range(8)], 1)]        # 7 another one
    ops += [("connect", 0, 2), ("connect", 2, 3), ("connect", 1, 3), ("connect", 0, 4), ("connect", 1, 4),
            ("connect", 3, 5), ("connect", 4, 5), ("connect", 5, 6), ("connect", 5, 7)]
    return ops


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, build
    build.build()
    api.lib()
    return api


@pytest.fixture(scope="module")
def gl():
    m = _load("test_general_layer")
    m.CASES = dict(m.CASES, kinds=circuit_kinds)
    return m


@pytest.fixture(scope="module")
def ctxs(api):
    c = {0: api.Context(0, api.GOLDILOCKS), 1: api.Context(0, api.BN254)}
    yield c
    gc.collect()  # verifiers and circuits go before the contexts they were made on
    for x in c.values():
        x.close()


CASES = ["mixed", "square", "one_gate", "random", "kinds"]


def host_verdict(api, gl, ops, field, claims, tr, inputs):
    """hg_gkr_verify on a host description, then every input claim against the input's MLE"""
    c = api.Circuit(None, field)
    gl.build(c, ops)
    try:
        cl = c.verify_gkr(claims, tr)
    except api.HgError:
        return False
    return all((api.mle_eval_host(field, vec, p.shape[0], p) == x).all() for vec, cc in zip(inputs, cl) for p, x in cc)


def verifier(api, gl, ctx, ops, field):
    desc = api.Circuit(None, field)
    gl.build(desc, ops)
    return api.GkrBatchVerifier(ctx, desc, MAX_BATCH)


def check_batches(api, gl, ops, field, bv, items):
    """items: (proof bytes, output claims, inputs); verified in batches of up to MAX_BATCH; returns the verdicts, which must equal
    the host verifier's"""
    got, want = [], []
    for s in range(0, len(items), MAX_BATCH):
        chunk = items[s:s + MAX_BATCH]
        res = bv.verify_batch([api.Keccak256Transcript.from_proof(p, field) for p, _, _ in chunk], [c for _, c, _ in chunk], [i for _, _, i in chunk])
        got += [ok for ok, _ in res]
        assert all(r == "" if ok else r != "" for ok, r in res)
        want += [host_verdict(api, gl, ops, field, c, api.Keccak256Transcript.from_proof(p, field), i) for p, c, i in chunk]
    assert got == want
    return got


def changed_input(gl, ins, field):
    bad = [x.copy() for x in ins]
    bad[0][0] = (int(bad[0][0]) + 1) % gl.PRIME[field] if field == 0 else bad[0][0] ^ 1
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("field", FIELDS)
def test_every_flip_of_restated_proofs(api, gl, oracle, ctxs, field, case):
    """The proof of the CPU restatement, the same proof under every single-element flip and the proof with a changed input, in
    batches of up to MAX_BATCH: the good proof is accepted, everything else rejected, as by the host verifier."""
    ops, oc, ins, claims = gl.make_instance(oracle, api, field, case)
    proof, _ = oc.prove_gkr(claims)
    flips = list(gl.element_flips(proof, field))
    items = [(proof, claims, ins)] + [(b, claims, ins) for b in flips] + [(proof, claims, changed_input(gl, ins, field))]
    bv = verifier(api, gl, ctxs[field], ops, field)
    assert check_batches(api, gl, ops, field, bv, items) == [True] + [False] * (len(flips) + 1)
    bv.free()


def shared_point_instances(api, gl, oracle, field, case, seeds):
    """inputs of several seeds with output claims at the points of seed 0 -> (ops, [(inputs, claims, the restatement's proof)])"""
    ops, _, _, claims0 = gl.make_instance(oracle, api, field, case, seed=seeds[0])
    nodes, outs = gl.node_shapes(ops)
    out = []
    for s in seeds:
        _, oc, ins, _ = gl.make_instance(oracle, api, field, case, seed=s)
        claims = [(pt, oracle.mle_eval(field, oc.value(o), pt.shape[0], pt)) for (pt, _), o in zip(claims0, outs)]
        out.append((ins, claims, oc.prove_gkr(claims)[0]))
    return ops, out


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("field", FIELDS)
def test_device_proofs_with_shared_points(api, gl, oracle, ctxs, field, case):
    """Proofs of four input sets made on the device (prefetch mode, the restatement's bytes) with output claims at the same points,
    so every weight and edge sum of the batch is shared, next to a flipped proof and a proof paired with another input set. In
    "kinds" the product and linear layers feed only the general layer, which leaves two claims on each of them: the prover has to
    budget their alpha challenges."""
    ctx = ctxs[field]
    ops, inst = shared_point_instances(api, gl, oracle, field, case, (0, 1, 2, 3))
    c = api.Circuit(ctx)
    gl.build(c, ops)
    items, pts = [], []
    for ins, claims, want in inst:
        c.evaluate_host(ins)
        tr = api.Keccak256Transcript(field)
        got = c.prove_gkr(claims, tr, api.MODE_PREFETCH)
        assert tr.into_proof() == want
        items.append((want, claims, ins))
        pts.append([p.tobytes() for cl in got for p, _ in cl])
    assert all(p == pts[0] for p in pts)  # the library's challenges do not depend on the proof: one point set for all
    flips = list(gl.element_flips(items[1][0], field))
    items.append((flips[len(flips) // 2], items[1][1], items[1][2]))
    items.append((items[0][0], items[0][1], items[1][2]))
    bv = verifier(api, gl, ctx, ops, field)
    assert check_batches(api, gl, ops, field, bv, items) == [True] * 4 + [False, False]
    bv.free()
    c.free()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["random", "kinds"])
@pytest.mark.parametrize("field", FIELDS)
def test_per_proof_points(api, gl, oracle, ctxs, field, case):
    """With an absorbing caller transcript every proof has its own points, so no quantity is shared: three device proofs are
    accepted, and when one of them is tampered with the others still are."""
    Absorbing = _load("test_gpu_verify").Absorbing
    ctx = ctxs[field]
    el = 2 if field == 0 else 4
    c = api.Circuit(ctx)
    items = []
    for seed in (1, 2, 3):
        ops, oc, ins, _ = gl.make_instance(oracle, api, field, case, seed=seed)
        if not items:
            gl.build(c, ops)
        nodes, outs = gl.node_shapes(ops)
        inner = Absorbing(field, seed)
        tr = api.CallbackTranscript(inner, field)
        claims = []
        for o in outs:
            pt = tr.squeeze_challenges((nodes[o][1] - 1).bit_length())
            claims.append((pt, oracle.mle_eval(field, oc.value(o), pt.shape[0], pt)))
        c.evaluate_host(ins)
        c.prove_gkr(claims, tr, api.MODE_INTERACTIVE)
        items.append((seed, claims, ins, inner.into_proof()))
    bv = verifier(api, gl, ctx, ops, field)

    def transcript(seed, claims, proof):
        tr = api.CallbackTranscript(Absorbing(field, seed, proof), field)
        for pt, _ in claims:
            assert (tr.squeeze_challenges(pt.shape[0]) == pt).all()
        return tr

    def run(tampered):
        proofs = [p for _, _, _, p in items]
        if tampered is not None:
            q = proofs[tampered].copy()
            k = el * (len(q) // el // 2)
            q[k] = (int(q[k]) + 1) % gl.PRIME[0] if field == 0 else q[k] ^ 1
            proofs[tampered] = q
        res = bv.verify_batch([transcript(s, cl, p) for (s, cl, _, _), p in zip(items, proofs)], [cl for _, cl, _, _ in items],
                              [i for _, _, i, _ in items])
        host = [host_verdict(api, gl, ops, field, cl, transcript(s, cl, p), i) for (s, cl, i, _), p in zip(items, proofs)]
        assert [ok for ok, _ in res] == host
        return host
    assert run(None) == [True, True, True]
    assert run(1) == [True, False, True]
    bv.free()
    c.free()


def large_layer_arrays(rng, p):
    """the S = 2^20 general layer of test_general_layer.py::test_large_general_layer_verifies (arity 2, num_reps 16, 2^15 gates
    per rep, one random product and one random add per gate, a constant on about a quarter of them)"""
    log2_sub, reps, ng = 15, 16, 1 << 15
    sub = 1 << log2_sub
    w = lambda k: rng.integers(0, sub, size=k)
    i0, i1, x0, x1 = rng.integers(0, 2, size=ng), rng.integers(0, 2, size=ng), w(ng), w(ng)
    coef = rng.integers(0, p, size=ng, dtype=np.uint64)
    has_const = rng.random(ng) < 0.25
    consts = rng.integers(0, p, size=ng, dtype=np.uint64)
    add_ptr = np.arange(ng + 1, dtype=np.uint64)
    mul_ptr = np.arange(ng + 1, dtype=np.uint64)
    return (2, log2_sub, reps, has_const.astype(np.uint8), consts, add_ptr, rng.integers(0, p, size=ng, dtype=np.uint64),
            rng.integers(0, 2, size=ng).astype(np.uint32), w(ng).astype(np.uint64), mul_ptr, coef, i0.astype(np.uint32), x0.astype(np.uint64),
            i1.astype(np.uint32), x1.astype(np.uint64))


@pytest.mark.gpu
def test_large_general_layer_in_a_batch(api, gl, oracle, ctxs):
    """Three device proofs of the S = 2^20 layer (Goldilocks) with the same claim point, and the first of them with a flipped
    phase-2 message: the batch accepts the three and rejects the fourth, as the host verifier does."""
    ctx, p = ctxs[0], gl.PRIME[0]
    rng = np.random.default_rng(5)
    arrays = large_layer_arrays(rng, p)
    log2_sub, reps, ng = arrays[1], arrays[2], len(arrays[3])
    n_in = reps << log2_sub

    def circuit(c):
        a, b = c.insert_input(log2_sub, reps), c.insert_input(log2_sub, reps)
        g = c.insert_vanilla_arrays(*arrays)
        c.connect(a, g)
        c.connect(b, g)
        return g
    c, h = api.Circuit(ctx), api.Circuit(None, api.GOLDILOCKS)
    g = circuit(c)
    circuit(h)
    nv = (ng * reps - 1).bit_length()
    pt = gl.rand_ext(0, rng, nv)
    items = []
    for _ in range(3):
        ins = [rng.integers(0, p, size=n_in, dtype=np.uint64) for _ in range(2)]
        c.evaluate_host(ins)
        ptr, n = c.node_value(g)
        claims = [(pt, oracle.mle_eval(0, api.NodeValueView(ctx, ptr, n).download(np.uint64, n), nv, pt))]
        tr = api.Keccak256Transcript()
        c.prove_gkr(claims, tr, api.MODE_PREFETCH)
        items.append((tr.into_proof(), claims, ins))
    # the proof: phase 1 (log2 S degree-2 rounds of two elements), X_k(u_lo) for k < 2, phase 2 (the same), X_k(v_lo);
    # the flip is the second element of phase 2's first round
    s_nv, esz = nv + 1, 16
    proof = items[0][0]
    assert len(proof) == (4 * s_nv + 4) * esz
    k = (2 * s_nv + 3) * esz
    items.append((proof[:k] + next(gl.element_flips(proof[k:], 0)), items[0][1], items[0][2]))
    bv = api.GkrBatchVerifier(ctx, h, 4)
    res = bv.verify_batch([api.Keccak256Transcript.from_proof(pr) for pr, _, _ in items], [cl for _, cl, _ in items], [i for _, _, i in items])
    host = []
    for pr, cl, ins in items:
        try:
            got = h.verify_gkr(cl, api.Keccak256Transcript.from_proof(pr))
            host.append(all((api.mle_eval_host(0, vec, q.shape[0], q) == x).all() for vec, cc in zip(ins, got) for q, x in cc))
        except api.HgError:
            host.append(False)
    assert [ok for ok, _ in res] == host == [True, True, True, False]
    bv.free()
    c.free()
