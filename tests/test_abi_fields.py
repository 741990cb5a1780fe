"""Field checks at the C ABI. Every handle belongs to one field (Goldilocks or BN254): an entry point keyed by a field id rejects
an unknown id, and one that takes two handles rejects a pair of different fields before it does any work. A host-only circuit
description keeps its non-throwing getters and refuses every call that needs a device."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = [0, 1]


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, build
    build.build()
    api.lib()
    return api


def prime(api, field):
    return api.GL_P if field == api.GOLDILOCKS else api.BN_R


def to_limbs(api, field, vals):
    """canonical integers -> little-endian u64 limbs, LIMBS[field] per element"""
    limbs = api.LIMBS[field]
    return np.array([(int(v) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for v in vals for j in range(limbs)], np.uint64)


def relay_circuit(api, field, ctx=None):
    """input (8 elements) -> out[j] = 3 * in[j]: one linear layer"""
    c = api.Circuit(ctx, field)
    i = c.insert_input(3)
    v = c.insert_vanilla(1, 3, [api.VanillaGate(adds=[(3, (0, j))]) for j in range(8)])
    c.connect(i, v)
    return c


def output_claim(api, field, x, seed):
    """a random point of the relay circuit's output and the output's MLE there (x: the input as integers)"""
    rng = np.random.default_rng(seed)
    p, el = prime(api, field), api.LIMBS[field] * api.DEGREE[field]
    r = to_limbs(api, field, [int(rng.integers(0, 2**62)) % p for _ in range(3 * api.DEGREE[field])]).reshape(3, el)
    y = to_limbs(api, field, [3 * v % p for v in x])
    return r, api.mle_eval_host(field, y, 3, r)


@pytest.mark.parametrize("bad", [2, -1])
def test_field_keyed_entry_points_reject_an_unknown_field_id(api, bad):
    L = api.lib()
    h = C.c_void_p()
    words = np.zeros(16, np.uint64)
    ptr = api._p(words)
    cb = lambda _user, _limbs: 0
    hooks = (api.SQUEEZE_FN(cb), api.WRITE_FN(cb), api.READ_FN(cb))
    calls = {
        "hg_transcript_new": lambda: L.hg_transcript_new(bad, C.byref(h)),
        "hg_transcript_from_proof": lambda: L.hg_transcript_from_proof(bad, ptr, 16, C.byref(h)),
        "hg_transcript_from_callbacks": lambda: L.hg_transcript_from_callbacks(bad, None, *hooks, 0, C.byref(h)),
        "hg_circuit_new_host": lambda: L.hg_circuit_new_host(bad, C.byref(h)),
        "hg_shard_merge": lambda: L.hg_shard_merge(bad, ptr, ptr, 4),
        "hg_mle_eval_host": lambda: L.hg_mle_eval_host(bad, ptr, 2, 1, ptr, ptr),
    }
    for name, call in calls.items():
        assert call() != 0, name
        assert L.hg_last_error().decode() == "unknown field id", name
        assert not h.value, name
    # the one query that answers for any id
    assert (L.hg_field_base_bytes(0), L.hg_field_base_bytes(1), L.hg_field_base_bytes(bad)) == (8, 32, 8)


@pytest.mark.parametrize("field", FIELDS)
def test_gkr_verify_rejects_a_transcript_of_the_other_field(api, field):
    c = relay_circuit(api, field)
    claim = output_claim(api, field, range(8), 0)
    with pytest.raises(api.HgError, match="transcript belongs to another field"):
        c.verify_gkr([claim], api.Keccak256Transcript.from_proof(b"\x00" * 64, 1 - field))
    # a transcript of the circuit's field gets past the check and runs out of proof
    with pytest.raises(api.HgError) as e:
        c.verify_gkr([claim], api.Keccak256Transcript.from_proof(b"", field))
    assert "another field" not in str(e.value)
    c.free()


@pytest.mark.parametrize("field", FIELDS)
def test_host_only_circuit_answers_getters_and_refuses_device_calls(api, field):
    L = api.lib()
    c = relay_circuit(api, field)
    assert c.shard_words == 0
    assert all(v == 0 for v in c.timing().values())   # the six phases and ext_challenges (hg_gkr_num_challenges)
    assert L.hg_gkr_input_claim_num_vars(c.h, 0, 0) == 0 and L.hg_gkr_num_inputs(c.h) == 0
    claim = output_claim(api, field, range(8), 1)
    words = np.zeros(64, np.uint64)
    p, n = C.c_void_p(), C.c_size_t(0)
    calls = {
        "hg_circuit_evaluate": lambda: api._chk(L.hg_circuit_evaluate(c.h, None, 0)),
        "hg_circuit_evaluate_host": lambda: c.evaluate_host([np.zeros(8 * api.LIMBS[field], np.uint64)]),
        "hg_circuit_node_value": lambda: api._chk(L.hg_circuit_node_value(c.h, 1, C.byref(p), C.byref(n))),
        "hg_gkr_prove": lambda: c.prove_gkr([claim], api.Keccak256Transcript(field)),
        "hg_gkr_prove_shard_dev": lambda: c.prove_gkr_shard_dev([claim], api.Keccak256Transcript(field), 0, 1, words.ctypes.data, words.size),
        "hg_gkr_emit_shard_dev": lambda: c.emit_shard_dev(words.ctypes.data, 0),
        "hg_gkr_emit_shard_part_dev": lambda: c.emit_shard_part_dev(words.ctypes.data, 0, 0, 1),
    }
    for name, call in calls.items():
        with pytest.raises(api.HgError, match="host-only"):
            call()
    c.free()


# ---- on the GPU: one context per field

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


def lasso_case(api, field, golden_dir):
    from hyper_greco_b200 import params, witness
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    tag, inputs = ("goldilocks", f"lasso_inputs_{name}.npz") if field == api.GOLDILOCKS else ("bn254", f"lasso_inputs_bn254_{name}.npz")
    inp = np.load(os.path.join(golden_dir, inputs))["inputs"]
    proof = open(os.path.join(golden_dir, f"proof_{tag}_lasso_node_{name}.bin"), "rb").read()
    return inp, witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P), proof


@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_mixed_field_pairs_are_rejected_before_any_work(api, ctxs, golden_dir, field):
    """A node, circuit or context of one field with a transcript (or Lasso node) of the other: an error, and no kernel is
    launched. Afterwards the context still proves correctly."""
    other = 1 - field
    ctx = ctxs(field)
    inp, bounds, segs, nv, golden_proof = lasso_case(api, field, golden_dir)
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx, pp, nv, segs)
    other_node = api.LassoNode(ctxs(other), pp, nv, segs)
    rng = np.random.default_rng(field)
    x = [int(v) for v in rng.integers(0, 2**62, size=8)]
    circuit = relay_circuit(api, field, ctx)
    circuit.evaluate_host([to_limbs(api, field, x)])
    r, val = output_claim(api, field, x, 2)
    el = api.LIMBS[field] * api.DEGREE[field]
    d_out = api.DeviceBuffer(ctx, 8 * max(node.shard_words, circuit.shard_words))
    d_tables = api.DeviceBuffer.from_field(ctx, to_limbs(api, field, x))
    coeffs, claim = to_limbs(api, field, [1] * api.DEGREE[field]), np.zeros(el, np.uint64)
    lasso_circuit = api.Circuit(ctx)
    wrong = lambda: api.Keccak256Transcript(other)
    calls = {
        "hg_lasso_node_prove": lambda: node.prove_claim_reduction(inp, wrong()),
        "hg_lasso_node_prove_shard": lambda: node.prove_shard(inp, wrong(), 0, 2),
        "hg_lasso_node_prove_shard_dev": lambda: node.prove_shard_dev(inp, wrong(), 0, 2, d_out.ptr, node.shard_words),
        "hg_gkr_prove": lambda: circuit.prove_gkr([(r, val)], wrong()),
        "hg_gkr_prove_shard_dev": lambda: circuit.prove_gkr_shard_dev([(r, val)], wrong(), 0, 1, d_out.ptr, circuit.shard_words),
        "hg_sumcheck_prove": lambda: api.sumcheck_prove(ctx, 1, coeffs, d_tables, 3, claim, wrong()),
        "hg_circuit_insert_lasso": lambda: lasso_circuit.insert_lasso(other_node),
    }
    ctx.synchronize()
    before = (ctx.launch_count, ctxs(other).launch_count)
    for name, call in calls.items():
        with pytest.raises(api.HgError, match="belongs to another field"):
            call()
    ctx.synchronize()
    assert (ctx.launch_count, ctxs(other).launch_count) == before

    # the context, the node and the circuit still prove correctly
    tr = api.Keccak256Transcript(field)
    node.prove_claim_reduction(inp, tr)
    assert tr.into_proof() == golden_proof
    tr = api.Keccak256Transcript(field)
    (claims,) = circuit.prove_gkr([(r, val)], tr)
    (pt, v), = claims
    assert (v == api.mle_eval_host(field, to_limbs(api, field, x), 3, pt)).all()
    host = relay_circuit(api, field)
    (vclaims,) = host.verify_gkr([(r, val)], api.Keccak256Transcript.from_proof(tr.into_proof(), field))
    assert len(vclaims) == 1 and (vclaims[0][0] == pt).all() and (vclaims[0][1] == v).all()
    for obj in (host, lasso_circuit, circuit, d_tables, d_out, other_node, node):
        obj.free()
