"""GPU parity tests (run with -m gpu on the B200 box). Everything goes through the C ABI (hyper_greco_b200.api ->
libhg_b200.so) and is compared bit-for-bit with the CPU oracle on the same inputs; at the BASELINE.json sizes the checks are
size-independent properties (oracle VERIFIER acceptance, claim == input MLE, prefetch == interactive, determinism)."""
import os

import numpy as np
import pytest

from conftest import load_case

pytestmark = pytest.mark.gpu
GL_P = 2**64 - 2**32 + 1


@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api
    api.lib()  # raises if the CUDA library is missing: no fallback
    return api


@pytest.fixture(scope="module")
def ctx(api):
    c = api.Context(0)
    yield c
    c.close()


def rand_ext(rng, n):
    return rng.integers(0, GL_P, size=(n, 2), dtype=np.uint64)


def test_device_field_arithmetic(api, ctx, oracle):
    rng = np.random.default_rng(0)
    edge = np.array([0, 1, GL_P - 1, GL_P - 2, 2**32, 2**32 - 1, 2**63, 0xFFFFFFFF00000000, 0xFFFFFFFF], np.uint64)
    a = np.concatenate([rand_ext(rng, 4096), np.stack(np.meshgrid(edge, edge), -1).reshape(-1, 2)])
    b = np.concatenate([rand_ext(rng, 4096), np.stack(np.meshgrid(edge, edge), -1).reshape(-1, 2)[::-1]])
    for op in (0, 1, 2):
        got = api.field_selftest(ctx, op, a, b)
        ai, bi = a.astype(object), b.astype(object)
        if op == 0:
            want = (ai + bi) % GL_P
        elif op == 1:
            want = (ai - bi) % GL_P
        else:
            want = np.stack([(ai[:, 0] * bi[:, 0] + 7 * ai[:, 1] * bi[:, 1]) % GL_P, (ai[:, 0] * bi[:, 1] + ai[:, 1] * bi[:, 0]) % GL_P], -1)
        assert (got.astype(object) == want).all(), op
    # and against the oracle's own arithmetic
    for i in range(0, 64):
        assert (api.field_selftest(ctx, 2, a[i:i + 1], b[i:i + 1])[0] == oracle.field_op(0, 2, a[i], b[i])).all()


FILLS = ("random", "max", "lazy_pairs")


def fill_params(shapes, fills=FILLS):
    """shape x fill; the random fill keeps the shape's own test id."""
    return [pytest.param(*sh, f, id="-".join(map(str, sh)) + ("" if f == "random" else "-" + f)) for f in fills for sh in shapes]


def fill_tables(rng, fill, shape, consts, rand):
    """Sumcheck inputs at the extremes, from consts = the elements (0, p - 2, p - 1) in the field's limb layout: `max` is every
    entry p - 1; `lazy_pairs` makes every pair (lo, hi) either (p - 1, p - 2) or (0, p - 1), whose line through the pair is p
    (a non-canonical zero) at X = -1 resp. takes the borrow at X = -1 and at infinity."""
    if fill == "random":
        return rand(shape)
    idx = np.full(shape, 2)
    if fill == "lazy_pairs":
        kind = rng.integers(0, 2, size=shape[:-1] + (shape[-1] // 2,))
        idx[..., 0::2] = np.where(kind == 0, 2, 0)
        idx[..., 1::2] = np.where(kind == 0, 1, 2)
    return consts[idx]


# the last shapes give more pairs than k_sc_round's grid (8 blocks of 256 threads per SM): every thread loops
SC_SHAPES = [(1, 2, 1), (1, 7, 4), (2, 1, 1), (2, 3, 2), (2, 5, 3), (2, 12, 11), (1, 25, 12), (2, 50, 9), (2, 2, 20), (1, 3, 20)]


@pytest.mark.parametrize("arity,nterms,nv,fill", fill_params(SC_SHAPES))
@pytest.mark.parametrize("mode", [0, 1])
def test_sumcheck_matches_oracle(api, ctx, oracle, arity, nterms, nv, fill, mode):
    rng = np.random.default_rng(nv * 100 + nterms)
    tables = fill_tables(rng, fill, (nterms * arity, 1 << nv), np.array([0, GL_P - 2, GL_P - 1], np.uint64),
                         lambda sh: rng.integers(0, GL_P, size=sh, dtype=np.uint64))
    coeffs = rand_ext(rng, nterms)
    claim = rand_ext(rng, 1)[0]
    if fill == "max":
        coeffs[:], claim[:] = GL_P - 1, GL_P - 1
    oproof, te, orr, ofe = oracle.sumcheck_prove(0, arity, coeffs, tables, nv, claim)
    d = api.DeviceBuffer.from_numpy(ctx, tables)
    t = api.Keccak256Transcript()
    pt, ev = api.sumcheck_prove(ctx, arity, coeffs, d, nv, claim, t, mode)
    assert t.into_proof() == oproof
    assert (pt == orr).all() and (ev == ofe).all()
    d.free()


@pytest.mark.parametrize("opts", [((3, 1),), ((31, 1),), ((3, 1), (31, 1))])
def test_sumcheck_wire_variants(api, oracle, opts):
    """Appendix-B switches A3 / A3': both implementations must agree under every setting."""
    rng = np.random.default_rng(5)
    arity, nterms, nv = 2, 4, 6
    tables = rng.integers(0, GL_P, size=(nterms * arity, 1 << nv), dtype=np.uint64)
    coeffs, claim = rand_ext(rng, nterms), rand_ext(rng, 1)[0]
    c = api.Context(0)
    try:
        for w, v in opts:
            oracle.set_assumption(w, v)
            c.set_option(w, v)
        oproof, *_ = oracle.sumcheck_prove(0, arity, coeffs, tables, nv, claim)
        d = api.DeviceBuffer.from_numpy(c, tables)
        t = api.Keccak256Transcript()
        api.sumcheck_prove(c, arity, coeffs, d, nv, claim, t)
        assert t.into_proof() == oproof
        d.free()
    finally:
        for w, v in ((3, 0), (31, 0), (5, 1)):
            oracle.set_assumption(w, v)
        c.close()


def _mle_cases(rng, rand_table, top_table, rand_point, edge_point):
    """(label, num_vars, n_tables, stride, tables [n_tables, stride], point). nv = 12 is where the low half of the eq split
    covers the whole table, nv = 21 where k_dot_eq's grid is capped at 2 blocks per SM; stride > 2^nv leaves gaps between
    the tables; several tables run as grid.y."""
    cases = []
    for nv in (1, 5, 13):
        cases.append((f"random nv={nv}", nv, 3, 1 << nv, rand_table((3, 1 << nv)), rand_point(nv)))
    for nv, nt, extra in ((12, 2, 0), (21, 2, 0), (7, 5, 10), (13, 4, 4096)):
        stride = (1 << nv) + extra
        cases.append((f"nv={nv} tables={nt} stride={stride}", nv, nt, stride, rand_table((nt, stride)), rand_point(nv)))
    for nv in (3, 12, 14):
        cases.append((f"max nv={nv}", nv, 2, 1 << nv, top_table((2, 1 << nv)), rand_point(nv)))
        cases.append((f"max at 0/1/p-1 point nv={nv}", nv, 2, 1 << nv, top_table((2, 1 << nv)), edge_point(rng, nv)))
        cases.append((f"random at 0/1/p-1 point nv={nv}", nv, 1, 1 << nv, rand_table((1, 1 << nv)), edge_point(rng, nv)))
    return cases


def test_mle_eval_batch_matches_oracle(api, ctx, oracle):
    rng = np.random.default_rng(9)
    edge = lambda rng, nv: rng.choice(np.array([0, 1, GL_P - 1], np.uint64), size=(nv, 2))
    for label, nv, nt, stride, tables, pt in _mle_cases(rng, lambda sh: rng.integers(0, GL_P, size=sh, dtype=np.uint64),
                                                        lambda sh: np.full(sh, GL_P - 1, np.uint64), lambda nv: rand_ext(rng, nv), edge):
        d = api.DeviceBuffer.from_numpy(ctx, tables)
        got = api.mle_eval_batch(ctx, d, nt, nv, pt, stride=stride)
        for i in range(nt):
            assert (got[i] == oracle.mle_eval(0, tables[i, :1 << nv], nv, pt)).all(), (label, i)
        d.free()
    # the tables are read with 16-byte vector loads: an odd stride is refused before any launch
    d = api.DeviceBuffer.from_numpy(ctx, np.zeros(2 * 17, np.uint64))
    with pytest.raises(api.HgError, match="aligned"):
        api.mle_eval_batch(ctx, d, 2, 4, rand_ext(rng, 4), stride=17)
    d.free()


def _prove_gpu(api, ctx, bounds, segs, nv, inp, mode=0, device_resident=False):
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx, pp, nv, segs)
    tr = api.Keccak256Transcript()
    if device_resident:
        buf = api.DeviceBuffer.from_numpy(ctx, inp)
        pt, val = node.prove_claim_reduction(buf, tr, mode, n_inputs=inp.size)
        buf.free()
    else:
        pt, val = node.prove_claim_reduction(inp, tr, mode)
    return node, pp, tr, pt, val


@pytest.mark.parametrize("name", ["1024_1x27_65537", "2048_1x52_65537", "4096_2x55_65537"])
@pytest.mark.parametrize("mode", [0, 1])
def test_lasso_node_proof_bytes_match_oracle_on_reference_fixtures(api, ctx, oracle, golden_dir, name, mode):
    P, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, golden_dir)
    oproof, orr, osum, nsq = oracle.lasso_prove(0, opp, nv, rows, inp)
    node, pp, tr, pt, val = _prove_gpu(api, ctx, bounds, segs, nv, inp, mode, device_resident=(mode == 0))
    assert tr.into_proof() == oproof
    assert tr.num_squeezed == nsq
    assert (pt.reshape(-1) == orr).all() and (val == osum).all()
    # polynomialised witness (lasso.rs:157-250)
    dims, rd, fc, e = node.download_polys()
    od, ord_, ofc, oe = oracle.lasso_polynomialize(0, opp, nv, rows, inp)
    assert (dims == od).all() and (e == oe).all()
    for slot, d in enumerate(sorted(set(opp.memory_to_dimension_index))):
        assert (rd[slot] == ord_[d]).all() and (fc[slot] == ofc[d]).all()
    # the reference's own acceptance test, on the GPU proof
    oracle.lasso_verify(0, opp, nv, tr.into_proof())
    assert node.log2_input_size() == max(nv, 16)
    node.free()


@pytest.mark.parametrize("opts", [((3, 1), (31, 1)), ((5, 0),)])
def test_lasso_node_under_assumption_switches(api, oracle, golden_dir, opts):
    P, inp, bounds, segs, nv, opp, rows = load_case("1024_1x27_65537", oracle, golden_dir)
    c = api.Context(0)
    try:
        for w, v in opts:
            oracle.set_assumption(w, v)
            c.set_option(w, v)
        oproof, *_ = oracle.lasso_prove(0, opp, nv, rows, inp)
        node, pp, tr, pt, val = _prove_gpu(api, c, bounds, segs, nv, inp)
        assert tr.into_proof() == oproof
        node.free()
    finally:
        for w, v in ((3, 0), (31, 0), (5, 1)):
            oracle.set_assumption(w, v)
        c.close()


def test_lasso_node_ragged_and_edge_inputs(api, ctx, oracle, golden_dir):
    """Edge cases the reference's structure implies: fewer inputs than lookups (izip stops early, Q9), values at the
    range boundaries, an out-of-range value (bits silently truncated, Q8), transcript offset (node not first in the proof)."""
    P, inp, bounds, segs, nv, opp, rows = load_case("1024_1x27_65537", oracle, golden_dir)
    cases = {"short": inp[: inp.size - 777].copy()}
    # an input whose padded length is not 2^num_vars trips assert_eq!(num_vars, self.num_vars) (lasso.rs:80) in both
    with pytest.raises(oracle.OracleError):
        oracle.lasso_prove(0, opp, nv, rows, inp[:1].copy())
    pp0 = api.LassoPreprocessing.preprocess(bounds)
    node0 = api.LassoNode(ctx, pp0, nv, segs)
    with pytest.raises(api.HgError):
        node0.prove_claim_reduction(inp[:1].copy(), api.Keccak256Transcript())
    node0.free()
    edge = inp.copy()
    edge[-1] = 65536          # k1 + K1_BOUND maximum
    edge[-2] = 0              # minimum
    edge[0] = 200000          # out of range for R1: truncated
    edge[5] = GL_P - 1        # a "negative" value that was not shifted into range
    cases["edge"] = edge
    for label, x in cases.items():
        oproof, orr, osum, _ = oracle.lasso_prove(0, opp, nv, rows, x)
        node, pp, tr, pt, val = _prove_gpu(api, ctx, bounds, segs, nv, x)
        assert tr.into_proof() == oproof, label
        assert (val == osum).all(), label
        node.free()
    # transcript already advanced by other nodes: skip 37 base squeezes = 18.5 -> use 38 (19 ext challenges)
    oproof, *_ = oracle.lasso_prove(0, opp, nv, rows, inp, skip=38)
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx, pp, nv, segs)
    tr = api.Keccak256Transcript()
    tr.squeeze_challenges(19)
    node.prove_claim_reduction(inp, tr)
    assert tr.into_proof() == oproof
    # a node can be reused for a second proof
    tr2 = api.Keccak256Transcript()
    tr2.squeeze_challenges(19)
    node.prove_claim_reduction(inp, tr2, 1)
    assert tr2.into_proof() == oproof
    node.free()


@pytest.mark.parametrize("name,seed", [("4096_2x55_65537", 11), ("8192_4x55_65537", 12)])
def test_lasso_node_synthetic_witness_matches_oracle(api, ctx, oracle, name, seed):
    P, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, seed=seed)
    oproof, orr, osum, _ = oracle.lasso_prove(0, opp, nv, rows, inp)
    node, pp, tr, pt, val = _prove_gpu(api, ctx, bounds, segs, nv, inp)
    assert tr.into_proof() == oproof
    node.free()


def test_lasso_node_full_size_properties(api, ctx, oracle):
    """BASELINE.json metric config: n=32768, k=16, Goldilocks (num_vars 21, 25 memories). The oracle prover needs minutes
    here, so parity is checked through size-independent properties: the oracle VERIFIER (restated from
    lasso/src/memory_checking/verifier.rs:130-235, lasso/src/lasso.rs:116-139) accepts the GPU proof; the returned claim is
    the MLE of the input at the squeezed point; prefetch and interactive modes give identical bytes; proving twice is
    deterministic; a flipped proof byte is rejected."""
    P, inp, bounds, segs, nv, opp, rows = load_case("32768_16x59_65537", oracle, seed=0)
    assert nv == 21 and opp.num_memories == 25
    node, pp, tr, pt, val = _prove_gpu(api, ctx, bounds, segs, nv, inp)
    proof = tr.into_proof()
    r, s, used = oracle.lasso_verify(0, opp, nv, proof)
    assert used == len(proof) and (r == pt.reshape(-1)).all() and (s == val).all()
    # the product's own host verifier (hg_lasso_node_verify) agrees with the oracle's
    vpt, vval = api.lasso_node_verify(pp, nv, api.Keccak256Transcript(api.GOLDILOCKS, proof))
    assert (vpt == pt).all() and (vval == val).all()
    padded = np.zeros(1 << nv, np.uint64)
    padded[: inp.size] = inp
    assert (oracle.mle_eval(0, padded, nv, pt.reshape(-1)) == val).all()
    tr2 = api.Keccak256Transcript()
    node.prove_claim_reduction(inp, tr2, 0)
    assert tr2.into_proof() == proof
    tr3 = api.Keccak256Transcript()
    node.prove_claim_reduction(inp, tr3, 1)
    assert tr3.into_proof() == proof
    bad = bytearray(proof)
    bad[-3] ^= 4
    with pytest.raises(oracle.OracleError):
        oracle.lasso_verify(0, opp, nv, bytes(bad))
    node.free()


def _prove_sharded_on_one_gpu(api, ctx, field, bounds, segs, nv, inp, world, skip_ext=0):
    """SURVEY.md §8e on one device: `world` node objects play the ranks; their message buffers are summed by hg_shard_merge
    and rank 0 serialises. The result must be the proof a single device writes."""
    pp = api.LassoPreprocessing.preprocess(bounds)
    nodes = [api.LassoNode(ctx, pp, nv, segs) for _ in range(world)]
    trs = [api.Keccak256Transcript(field) for _ in range(world)]
    parts = []
    for r in range(world):
        if skip_ext:
            trs[r].squeeze_challenges(skip_ext)
        parts.append(nodes[r].prove_shard(inp, trs[r], r, world).copy())
    # slots are owned by exactly one rank or are sums: ranks other than 0 leave most slots zero
    assert all(p.size == parts[0].size for p in parts)
    merged = parts[0].copy()
    for r in range(1, world):
        api.shard_merge(field, merged, parts[r])
    pt, val = nodes[0].emit_shard(merged)
    proof = trs[0].into_proof()
    for n in nodes:
        n.free()
    return proof, pt, val, parts


@pytest.mark.parametrize("name,world", [("1024_1x27_65537", 2), ("2048_1x52_65537", 3), ("4096_2x55_65537", 4), ("4096_2x55_65537", 8)])
def test_lasso_node_sharded_proof_equals_single_device_proof(api, ctx, oracle, golden_dir, name, world):
    P, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, golden_dir)
    oproof, orr, osum, _ = oracle.lasso_prove(0, opp, nv, rows, inp)
    proof, pt, val, parts = _prove_sharded_on_one_gpu(api, ctx, api.GOLDILOCKS, bounds, segs, nv, inp, world)
    assert proof == oproof
    assert (pt.reshape(-1) == orr).all() and (val == osum).all()
    # the work really is split: every rank contributes, and no rank alone holds the whole buffer
    for p in parts:
        assert p.any()
        assert (p == 0).sum() > p.size // (2 * world)
    # a shard followed by an ordinary proof on the same node still gives the single-device bytes
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx, pp, nv, segs)
    node.prove_shard(inp, api.Keccak256Transcript(), 1, world)
    tr = api.Keccak256Transcript()
    node.prove_claim_reduction(inp, tr)
    assert tr.into_proof() == oproof
    with pytest.raises(api.HgError):
        node.prove_shard(inp, api.Keccak256Transcript(), world, world)
    node.free()


def test_lasso_node_sharded_full_size_and_offset(api, ctx, oracle):
    """Full-size node (num_vars 21, 25 memories, 50 vectors) over 4 ranks with an advanced transcript == one device."""
    P, inp, bounds, segs, nv, opp, rows = load_case("32768_16x59_65537", oracle, seed=0)
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx, pp, nv, segs)
    tr = api.Keccak256Transcript()
    tr.squeeze_challenges(7)
    node.prove_claim_reduction(inp, tr)
    node.free()
    proof, pt, val, _ = _prove_sharded_on_one_gpu(api, ctx, api.GOLDILOCKS, bounds, segs, nv, inp, 4, skip_ext=7)
    assert proof == tr.into_proof()


def test_bn254_lasso_node_sharded(api, ctx_bn, oracle, golden_dir):
    import os
    from hyper_greco_b200 import params, witness
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    inp = np.load(os.path.join(golden_dir, f"lasso_inputs_bn254_{name}.npz"))["inputs"]
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    opp = oracle.Preprocessing(bounds)
    rows = np.concatenate([np.full(l, opp.lookup_index(b), np.int32) for b, l in segs])
    oproof, *_ = oracle.lasso_prove(1, opp, nv, rows, inp)
    proof, pt, val, _ = _prove_sharded_on_one_gpu(api, ctx_bn, api.BN254, bounds, segs, nv, inp, 2)
    assert proof == oproof


def ntt_fill(rng, fill, shape, top, rand):
    """NTT inputs at the extremes: all top (= p - 1), a single top in zeros, or the powers of 2^32 mod p (0, 2^32, 2^64 - 2^32 ...)."""
    if fill == "random":
        return rand(shape)
    x = np.zeros(shape, dtype=object)
    if fill == "max":
        x[...] = top
    elif fill == "single_max":
        x[..., rng.integers(0, shape[-1])] = top
    else:
        x[...] = [pow(2, 32 * (j % 6), top + 1) for j in range(shape[-1])]
    return x


NTT_SHAPES = [(1, 3), (2, 1), (5, 4), (8, 2), (11, 3), (13, 2), (16, 3), (17, 1)]


@pytest.mark.parametrize("log_n,batch,fill", fill_params(NTT_SHAPES, ("random",)) +
                         fill_params([(1, 3), (5, 4), (11, 3), (16, 3)], ("max", "single_max", "pow2_32")))
def test_ntt_matches_oracle(api, ctx, oracle, log_n, batch, fill):
    """FftNode forward / inverse evaluation (assumption A9: natural order, inverse scaled by 1/n)."""
    rng = np.random.default_rng(log_n)
    x = ntt_fill(rng, fill, (batch, 1 << log_n), GL_P - 1, lambda sh: rng.integers(0, GL_P, size=sh, dtype=np.uint64)).astype(np.uint64)
    for inverse in (False, True):
        d = api.DeviceBuffer.from_numpy(ctx, x)
        api.ntt(ctx, d, log_n, inverse, batch)
        got = d.download(np.uint64, x.size).reshape(x.shape)
        assert (got == oracle.ntt(0, x, log_n, inverse)).all(), (log_n, inverse)
        d.free()
    # size-independent properties: inverse(forward(x)) = x, and the transform of a delta at 1 is the root powers
    d = api.DeviceBuffer.from_numpy(ctx, x)
    api.ntt(ctx, d, log_n, False, batch)
    api.ntt(ctx, d, log_n, True, batch)
    assert (d.download(np.uint64, x.size).reshape(x.shape) == x).all()
    d.free()


@pytest.mark.parametrize("name", ["1024_1x27_65537", "4096_2x55_65537"])
def test_bfv_forward_evaluation_on_reference_fixture(api, ctx, oracle, golden_dir, name):
    """circuit.evaluate on the reference's own witness: the `sum` layer equals ct0is (the circuit identity the reference's
    verify() relies on, sk_encryption_circuit.rs:512-516) and the `lasso_inputs_batched` layer equals the golden vector; the
    Lasso node then proves straight from the device-resident layer."""
    import os
    from hyper_greco_b200 import params
    P = params.PARAMS[name]
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    want_lasso = np.load(os.path.join(golden_dir, f"lasso_inputs_{name}.npz"))["inputs"]
    bfv = api.BfvEncrypt(ctx, P)
    dev = bfv.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    lasso, summ = bfv.evaluate(dev)
    assert (lasso.download(np.uint64, want_lasso.size) == want_lasso).all()
    assert (summ.download(np.uint64, io["ct0is"].size) == io["ct0is"]).all()
    # oracle agrees on the same layers
    ins = {k: [int(v) for v in io[k]] for k in ("s", "e", "k1", "r2is")}
    ins["ais"] = [[int(v) for v in row] for row in io["ais"]]
    ins["r1is"] = [[int(v) for v in row] for row in io["r1is"]]
    ol, osum = oracle.bfv_eval(0, P, ins)
    assert (ol == want_lasso).all() and (osum == io["ct0is"]).all()
    # prove from the device-resident layer
    _, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, golden_dir)
    oproof, *_ = oracle.lasso_prove(0, opp, nv, rows, inp)
    tr = api.Keccak256Transcript()
    bfv.node.prove_claim_reduction(lasso, tr, n_inputs=want_lasso.size)
    assert tr.into_proof() == oproof


def test_bfv_forward_evaluation_full_size(api, ctx):
    """n=32768, k=16: 33 transforms of 2^16; the sum layer must equal ct0is of the synthetic witness."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(32768)
    args = witness.synth_witness(P, 3)
    ins, ct0is = witness.get_inputs(P, args)
    bfv = api.BfvEncrypt(ctx, P)
    lasso, summ = bfv.evaluate(bfv.upload_inputs(ins))
    assert (summ.download(np.uint64, len(ct0is)) == np.array(ct0is, dtype=np.uint64)).all()
    want = np.array(witness.lasso_inputs(P, args), dtype=np.uint64)
    assert (lasso.download(np.uint64, want.size) == want).all()


def _circuit_io(golden_dir, name):
    import os
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    ins = {k: [int(v) for v in io[k]] for k in ("s", "e", "k1", "r2is")}
    ins["ais"] = [[int(v) for v in row] for row in io["ais"]]
    ins["r1is"] = [[int(v) for v in row] for row in io["r1is"]]
    return io, ins, [int(v) for v in io["ct0is"]]


@pytest.mark.parametrize("name", ["1024_1x27_65537", "4096_2x55_65537"])
@pytest.mark.parametrize("mode", [0, 1])
def test_full_gkr_prove_matches_oracle_on_reference_fixtures(api, ctx, oracle, golden_dir, name, mode):
    """BfvEncrypt::prove (sk_encryption_circuit.rs:417-460) end to end on the device: every Vanilla / FFT / Lasso node. The proof
    bytes equal the CPU restatement's, its verifier (verify_gkr + the input-claim check of :512-516) accepts, and every returned
    input claim equals the MLE of the corresponding input at the claim point."""
    from hyper_greco_b200 import params
    P = params.PARAMS[name]
    io, ins, ct0is = _circuit_io(golden_dir, name)
    oproof = oracle.bfv_prove(0, P, ins, ct0is)
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    d_ct = api.DeviceBuffer.from_numpy(ctx, io["ct0is"])
    proof, claims = prover.prove(dev, d_ct, mode)
    assert proof == oproof
    oracle.bfv_verify(0, P, ins, ct0is, proof)
    flat = [io["s"], io["e"], io["k1"]] + list(io["ais"]) + list(io["r1is"]) + [io["r2is"]]
    assert len(claims) == len(flat)
    for vec, cl in zip(flat, claims):
        assert len(cl) >= 1
        for pt, v in cl:
            assert (oracle.mle_eval(0, np.asarray(vec, np.uint64), pt.shape[0], pt) == v).all()
    # forward evaluation kept on the device: the sum layer equals ct0is
    ptr, n = prover.circuit.node_value(prover.ids["sum"])
    assert n == io["ct0is"].size
    # BfvEncrypt::prove from host vectors (uploads + level-batched evaluate inside): the same bytes, twice (buffers are reused)
    for _ in range(2):
        proof_h, claims_h = prover.prove_host(flat, io["ct0is"], mode)
        assert proof_h == oproof
    assert all((a[0][1] == b[0][1]).all() for a, b in zip(claims, claims_h))
    with pytest.raises(api.HgError):
        prover.circuit.evaluate_host(flat[:-1])


def test_full_gkr_prove_full_size_properties(api, ctx, oracle):
    """n=32768, k=16: the oracle prover needs ~30 s here, so the full-size check is through properties: the oracle VERIFIER
    accepts the device proof (all layer sumchecks, the Lasso node, the input-claim check), and prefetch == interactive bytes."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(32768)
    args = witness.synth_witness(P, 5)
    ins, ct0is = witness.get_inputs(P, args)
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs(ins)
    d_ct = api.DeviceBuffer.from_numpy(ctx, np.array(ct0is, dtype=np.uint64))
    proof, claims = prover.prove(dev, d_ct, 0)
    oracle.bfv_verify(0, P, ins, ct0is, proof)
    proof2, _ = prover.prove(dev, d_ct, 0)
    assert proof2 == proof
    flat = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
    proof3, _ = prover.prove_host([np.array(v, dtype=np.uint64) for v in flat], np.array(ct0is, dtype=np.uint64), 0)
    assert proof3 == proof
    # the PRODUCT's own host verifier (hg_gkr_verify, no GPU involved) agrees with the oracle's: accepts, same input claims; rejects a flip
    ver = api.BfvSkEncryptVerifier(P)
    hflat = [np.array(v, dtype=np.uint64) for v in flat]
    vclaims = ver.verify(hflat, np.array(ct0is, dtype=np.uint64), proof)
    assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for ca, cb in zip(claims, vclaims) for a, b in zip(ca, cb))
    bad = bytearray(proof)
    bad[40] ^= 2
    with pytest.raises(api.HgError):
        ver.verify(hflat, np.array(ct0is, dtype=np.uint64), bytes(bad))


def test_full_gkr_prove_n16384_k8(api, ctx, oracle):
    """BASELINE.json config 3 (n=16384, log q=54, k=8, Goldilocks): whole BfvEncrypt::prove from host vectors; the oracle
    verifier accepts, every input claim is the MLE of its input, prefetch and interactive modes agree."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(16384)
    args = witness.synth_witness(P, 3)
    ins, ct0is = witness.get_inputs(P, args)
    flat = [np.array(v, dtype=np.uint64) for v in [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]]
    prover = api.BfvSkEncryptProver(ctx, P)
    proof, claims = prover.prove_host(flat, np.array(ct0is, dtype=np.uint64), 0)
    oracle.bfv_verify(0, P, ins, ct0is, proof)
    for vec, cl in zip(flat, claims):
        for pt, v in cl:
            assert (oracle.mle_eval(0, vec, pt.shape[0], pt) == v).all()
    proof_i, _ = prover.prove_host(flat, np.array(ct0is, dtype=np.uint64), 1)
    assert proof_i == proof


# ------------------------------------------------------------------------------------------------ BN254 Fr (E = F)
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


@pytest.fixture(scope="module")
def ctx_bn(api):
    c = api.Context(0, api.BN254)
    yield c
    c.close()


def rand_fr_limbs(rng, shape):
    """Canonical limbs of uniform-ish elements (a top limb below r's is enough), vectorised for large tables."""
    t = rng.integers(0, 2**64, size=tuple(shape) + (4,), dtype=np.uint64)
    t[..., 3] %= np.uint64(BN_R >> 192)
    return t


def rand_fr_int(rng, shape):
    return np.array([int.from_bytes(rng.bytes(40), "little") % BN_R for _ in range(int(np.prod(shape)))], dtype=object).reshape(shape)


def rand_fr(rng, shape):
    vals = rand_fr_int(rng, shape).reshape(-1)
    return np.array([[(v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for v in vals], dtype=np.uint64).reshape(*shape, 4)


def test_bn254_device_field_arithmetic(api, ctx_bn, oracle):
    rng = np.random.default_rng(1)
    a, b = rand_fr(rng, (300,)), rand_fr(rng, (300,))
    edge = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0x43e1f593f0000000, 0x2833e84879b97091, 0xb85045b68181585d, 0x30644e72e131a029]], np.uint64)
    a[:3], b[:3] = edge, edge[::-1]
    to_int = lambda l: [sum(int(x[j]) << (64 * j) for j in range(4)) for x in l]
    ai, bi = to_int(a), to_int(b)
    for op, f in ((0, lambda x, y: (x + y) % BN_R), (1, lambda x, y: (x - y) % BN_R), (2, lambda x, y: x * y % BN_R)):
        got = to_int(api.field_selftest(ctx_bn, op, a, b))
        assert got == [f(x, y) for x, y in zip(ai, bi)], op


@pytest.mark.parametrize("arity,nterms,nv,fill", fill_params([(1, 3, 4), (2, 1, 1), (2, 4, 7), (2, 6, 3), (2, 1, 20)]))
@pytest.mark.parametrize("mode", [0, 1])
def test_bn254_sumcheck_matches_oracle(api, ctx_bn, oracle, arity, nterms, nv, fill, mode):
    rng = np.random.default_rng(nv * 10 + nterms)
    tables = fill_tables(rng, fill, (nterms * arity, 1 << nv), _bn_limbs([0, BN_R - 2, BN_R - 1]),
                         lambda sh: rand_fr(rng, sh) if np.prod(sh) <= 1 << 16 else rand_fr_limbs(rng, sh))
    coeffs, claim = rand_fr(rng, (nterms,)), rand_fr(rng, (1,))[0]
    if fill == "max":
        coeffs, claim = _bn_limbs([BN_R - 1] * nterms), _bn_limbs([BN_R - 1])[0]
    oproof, te, orr, ofe = oracle.sumcheck_prove(1, arity, coeffs, tables, nv, claim)
    d = api.DeviceBuffer.from_field(ctx_bn, tables)
    t = api.Keccak256Transcript(api.BN254)
    pt, ev = api.sumcheck_prove(ctx_bn, arity, coeffs, d, nv, claim, t, mode)
    assert t.into_proof() == oproof
    assert (pt == orr).all() and (ev == ofe).all()
    d.free()


@pytest.mark.parametrize("name", ["1024_1x27_65537", "2048_1x52_65537"])
@pytest.mark.parametrize("mode", [0, 1])
def test_bn254_lasso_node_proof_bytes_match_oracle(api, ctx_bn, oracle, golden_dir, name, mode):
    """The reference's BN254 witnesses (bfv-gkr/src/data/bn254): Lasso node proof bytes == oracle, oracle verifier accepts."""
    import os
    from hyper_greco_b200 import params, witness
    P = params.PARAMS[name]
    inp = np.load(os.path.join(golden_dir, f"lasso_inputs_bn254_{name}.npz"))["inputs"]
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    opp = oracle.Preprocessing(bounds)
    rows = np.concatenate([np.full(l, opp.lookup_index(b), np.int32) for b, l in segs])
    oproof, orr, osum, nsq = oracle.lasso_prove(1, opp, nv, rows, inp)
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx_bn, pp, nv, segs)
    tr = api.Keccak256Transcript(api.BN254)
    if mode == 0:
        buf = api.DeviceBuffer.from_field(ctx_bn, inp)
        pt, val = node.prove_claim_reduction(buf, tr, mode, n_inputs=inp.shape[0])
    else:
        pt, val = node.prove_claim_reduction(inp, tr, mode)
    assert tr.into_proof() == oproof
    assert tr.num_squeezed == nsq
    assert (pt.reshape(-1) == orr).all() and (val == osum).all()
    oracle.lasso_verify(1, opp, nv, tr.into_proof())
    dims, rd, fc, e = node.download_polys()
    od, ord_, ofc, oe = oracle.lasso_polynomialize(1, opp, nv, rows, inp)
    assert (dims == od).all() and (e == oe).all()
    node.free()


@pytest.mark.parametrize("mode", [0, 1])
def test_bn254_full_gkr_prove_matches_oracle(api, ctx_bn, oracle, golden_dir, mode):
    """BfvEncrypt::prove over BN254 Fr (E = F) on the reference's own BN254 witness (bfv-gkr/src/data/bn254, n=1024): every
    node of the circuit on the device, from host vectors; proof bytes == oracle, oracle verifier accepts."""
    import os
    from hyper_greco_b200 import params
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    io = np.load(os.path.join(golden_dir, f"circuit_io_bn254_{name}.npz"))
    ints = lambda a: [sum(int(r[j]) << (64 * j) for j in range(4)) for r in a.reshape(-1, 4)]
    ins = dict(s=ints(io["s"]), e=ints(io["e"]), k1=ints(io["k1"]), ais=[ints(a) for a in io["ais"]], r1is=[ints(a) for a in io["r1is"]],
               r2is=ints(io["r2is"]))
    ct0is = ints(io["ct0is"])
    oproof = oracle.bfv_prove(1, P, ins, ct0is)
    oracle.bfv_verify(1, P, ins, ct0is, oproof)
    prover = api.BfvSkEncryptProver(ctx_bn, P)
    flat = [io["s"], io["e"], io["k1"]] + list(io["ais"]) + list(io["r1is"]) + [io["r2is"]]
    proof, claims = prover.prove_host([np.ascontiguousarray(v).reshape(-1) for v in flat], io["ct0is"].reshape(-1), mode)
    assert proof == oproof
    oracle.bfv_verify(1, P, ins, ct0is, proof)
    assert len(claims) == len(flat)


def test_device_proofs_equal_committed_oracle_generated_golden_bytes(api, ctx, ctx_bn, golden_dir):
    """Device output against the COMMITTED proof bytes (tests/golden/golden_proofs.json), without the oracle in the loop:
    Lasso node and whole BfvEncrypt::prove, Goldilocks and BN254, on the reference's n=1024 witnesses."""
    import hashlib
    import json
    import os
    from hyper_greco_b200 import params, witness
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    meta = json.load(open(os.path.join(golden_dir, "golden_proofs.json")))["files"]

    def golden(fname):
        data = open(os.path.join(golden_dir, fname), "rb").read()
        assert hashlib.sha256(data).hexdigest() == meta[fname]["sha256"]
        return data

    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    for field, c, tag, lasso_file, io_file in ((api.GOLDILOCKS, ctx, "goldilocks", f"lasso_inputs_{name}.npz", f"circuit_io_{name}.npz"),
                                               (api.BN254, ctx_bn, "bn254", f"lasso_inputs_bn254_{name}.npz", f"circuit_io_bn254_{name}.npz")):
        inp = np.load(os.path.join(golden_dir, lasso_file))["inputs"]
        node = api.LassoNode(c, api.LassoPreprocessing.preprocess(bounds), nv, segs)
        tr = api.Keccak256Transcript(field)
        node.prove_claim_reduction(inp, tr)
        assert tr.into_proof() == golden(f"proof_{tag}_lasso_node_{name}.bin"), tag
        node.free()
        io = np.load(os.path.join(golden_dir, io_file))
        flat = [io["s"], io["e"], io["k1"]] + list(io["ais"]) + list(io["r1is"]) + [io["r2is"]]
        prover = api.BfvSkEncryptProver(c, P)
        proof, _ = prover.prove_host([np.ascontiguousarray(v).reshape(-1) for v in flat], np.ascontiguousarray(io["ct0is"]).reshape(-1))
        assert proof == golden(f"proof_{tag}_bfv_encrypt_{name}.bin"), tag


def test_bn254_ntt_matches_oracle(api, ctx_bn, oracle):
    rng = np.random.default_rng(2)
    cases = [(log_n, "random") for log_n in (3, 10, 13)] + [(log_n, f) for log_n in (3, 10) for f in ("max", "single_max", "pow2_32")]
    for log_n, fill in cases:
        x = _bn_limbs(ntt_fill(rng, fill, (2, 1 << log_n), BN_R - 1, lambda sh: rand_fr_int(rng, sh)).reshape(-1)).reshape(2, 1 << log_n, 4)
        for inverse in (False, True):
            d = api.DeviceBuffer.from_field(ctx_bn, x)
            api.ntt(ctx_bn, d, log_n, inverse, 2)
            got = d.to_field(2 << log_n).reshape(x.shape)
            assert (got == oracle.ntt(1, x, log_n, inverse).reshape(x.shape)).all(), (log_n, fill, inverse)
            d.free()


def test_bn254_mle_eval_batch_matches_oracle(api, ctx_bn, oracle):
    rng = np.random.default_rng(19)
    edge = lambda rng, nv: _bn_limbs(rng.choice(np.array([0, 1, BN_R - 1], dtype=object), size=nv))
    top = lambda sh: np.broadcast_to(_bn_limbs([BN_R - 1])[0], sh + (4,)).copy()
    for label, nv, nt, stride, tables, pt in _mle_cases(rng, lambda sh: rand_fr_limbs(rng, sh), top, lambda nv: rand_fr(rng, (nv,)), edge):
        d = api.DeviceBuffer.from_field(ctx_bn, tables)
        got = api.mle_eval_batch(ctx_bn, d, nt, nv, pt, stride=stride)
        for i in range(nt):
            assert (got[i] == oracle.mle_eval(1, tables[i, :1 << nv], nv, pt)).all(), (label, i)
        d.free()


# ------------------------------------------------------------------------------------------------ full-size byte parity
def _fullsize_meta(golden_dir, key):
    import json
    import os
    meta = json.load(open(os.path.join(golden_dir, "golden_proofs.json"))).get("fullsize", {})
    if key not in meta:
        pytest.skip(f"{key} not generated yet (tests/golden/make_golden_fullsize.py)")
    return meta[key]


def _assert_hash(proof, meta, what):
    import hashlib
    assert len(proof) == meta["bytes"], what
    assert hashlib.sha256(proof).hexdigest() == meta["sha256"], f"{what}: device proof bytes differ from the CPU oracle's (committed sha256)"


def test_fullsize_lasso_node_bytes_equal_oracle_hash(api, ctx, golden_dir):
    """BASELINE.json config 4 (n=32768, k=16, Goldilocks): the Lasso node's proof BYTES equal the CPU oracle's, through the
    committed sha256 (tests/golden/make_golden_fullsize.py). Host input and device-resident input, prefetch mode; interactive too."""
    from hyper_greco_b200 import params, witness
    meta = _fullsize_meta(golden_dir, "goldilocks_lasso_node_n32768_seed0")
    P = params.by_n(32768)
    inp = np.array(witness.lasso_inputs(P, witness.synth_witness(P, 0)), dtype=np.uint64)
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    node, pp, tr, pt, val = _prove_gpu(api, ctx, bounds, segs, nv, inp, 0, device_resident=True)
    _assert_hash(tr.into_proof(), meta, "lasso node n=32768 (prefetch)")
    tr = api.Keccak256Transcript()
    node.prove_claim_reduction(inp, tr, 1)
    _assert_hash(tr.into_proof(), meta, "lasso node n=32768 (interactive)")
    node.free()


@pytest.mark.parametrize("n,seed", [(32768, 5), (16384, 3)])
def test_fullsize_bfv_encrypt_bytes_equal_oracle_hash(api, ctx, golden_dir, n, seed):
    """BASELINE.json configs 3 and 4: whole BfvEncrypt::prove from HOST vectors (prove_host: H2D, evaluate, output claim,
    prove_gkr) gives the CPU oracle's bytes at n=16384 k=8 and n=32768 k=16."""
    from hyper_greco_b200 import params, witness
    meta = _fullsize_meta(golden_dir, f"goldilocks_bfv_encrypt_n{n}_seed{seed}")
    P = params.by_n(n)
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, seed))
    flat = [np.array(v, dtype=np.uint64) for v in [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]]
    prover = api.BfvSkEncryptProver(ctx, P)
    proof, _ = prover.prove_host(flat, np.array(ct0is, dtype=np.uint64), 0)
    _assert_hash(proof, meta, f"BfvEncrypt::prove n={n}")
    prover.circuit.free()
    prover.lasso.free()


def _bn_limbs(vals):
    return np.array([[(int(v) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for v in vals], dtype=np.uint64)


def test_fullsize_bn254_bytes_equal_oracle_hash(api, ctx_bn, oracle, golden_dir):
    """BASELINE.json config 5 (n=32768, k=16, BN254 Fr): Lasso node and whole BfvEncrypt::prove against the CPU oracle's
    sha256; the oracle verifier accepts the device proof of the node."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(32768)
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    meta = _fullsize_meta(golden_dir, "bn254_lasso_node_n32768_seed0")
    inp = _bn_limbs(witness.lasso_inputs(P, witness.synth_witness(P, 0, p=witness.BN_R), p=witness.BN_R))
    pp = api.LassoPreprocessing.preprocess(bounds)
    node = api.LassoNode(ctx_bn, pp, nv, segs)
    tr = api.Keccak256Transcript(api.BN254)
    node.prove_claim_reduction(inp, tr, 0)
    proof = tr.into_proof()
    node.free()
    _assert_hash(proof, meta, "bn254 lasso node n=32768")
    oracle.lasso_verify(1, oracle.Preprocessing(bounds), nv, proof)
    meta = _fullsize_meta(golden_dir, "bn254_bfv_encrypt_n32768_seed5")
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, 5, p=witness.BN_R))
    flat = [_bn_limbs(v).reshape(-1) for v in [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]]
    prover = api.BfvSkEncryptProver(ctx_bn, P)
    proof, _ = prover.prove_host(flat, _bn_limbs(ct0is).reshape(-1), 0)
    _assert_hash(proof, meta, "bn254 BfvEncrypt::prove n=32768")
    prover.circuit.free()
    prover.lasso.free()


# ------------------------------------------------------------------------------------------------ caller-owned transcript
@pytest.mark.parametrize("independent", [False, True])
def test_lasso_node_with_callback_transcript(api, ctx, golden_dir, independent):
    """hg_transcript_from_callbacks: the `&mut dyn TranscriptWrite<F, E>` of Node::prove_claim_reduction (lasso.rs:58-63) as C
    callbacks. The library is asked for prefetch mode; a transcript that may absorb messages forces the interactive schedule
    (squeezes interleaved with writes, in protocol order), one declared message-independent is prefetched (all squeezes of the
    node first). Either way the bytes the CALLER's transcript ends up with are the committed golden proof."""
    import os
    from hyper_greco_b200 import params, witness
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    golden = open(os.path.join(golden_dir, f"proof_goldilocks_lasso_node_{name}.bin"), "rb").read()
    inp = np.load(os.path.join(golden_dir, f"lasso_inputs_{name}.npz"))["inputs"]
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    node = api.LassoNode(ctx, api.LassoPreprocessing.preprocess(bounds), nv, segs)
    tr = api.CallbackTranscript(api.Keccak256Transcript(), message_independent=independent)
    pt, val = node.prove_claim_reduction(inp, tr, api.MODE_PREFETCH)
    assert tr.into_proof() == golden
    kinds = [k for k, _ in tr.log]
    n_sq, first_write = kinds.count("squeeze"), kinds.index("write")
    assert kinds.count("write") * 16 == len(golden)
    if independent:
        assert first_write == n_sq                      # every challenge of the node was squeezed before the first message
    else:
        assert first_write == nv                        # r (lasso.rs:85), then the claimed sum (:269): strictly protocol order
        assert "squeeze" in kinds[first_write:]         # and challenges keep coming between messages
    assert [tuple(int(x) for x in p) for p in pt] == [v for k, v in tr.log if k == "squeeze"][:nv]
    # a callback that fails surfaces as an error, not as a crash
    class Failing(api.Keccak256Transcript):
        def write_felt_ext(self, e):
            raise RuntimeError("sink is full")
    with pytest.raises(api.HgError):
        node.prove_claim_reduction(inp, api.CallbackTranscript(Failing()), api.MODE_PREFETCH)
    tr2 = api.Keccak256Transcript()                     # the node is still usable afterwards
    node.prove_claim_reduction(inp, tr2, api.MODE_PREFETCH)
    assert tr2.into_proof() == golden
    node.free()


def test_full_gkr_prove_with_callback_transcript(api, ctx, golden_dir):
    """gkr::prove_gkr of the whole circuit with a caller-owned transcript (interactive schedule): committed golden bytes."""
    import os
    from hyper_greco_b200 import params
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    golden = open(os.path.join(golden_dir, f"proof_goldilocks_bfv_encrypt_{name}.bin"), "rb").read()
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    d_ct = api.DeviceBuffer.from_numpy(ctx, io["ct0is"])
    prover.circuit.evaluate(dev)
    tr = api.CallbackTranscript(api.Keccak256Transcript())
    L = prover.ct0is_log2_size
    point = tr.squeeze_challenges(L)
    value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
    el = point.shape[1]
    prover.circuit.prove_gkr([(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)], tr, api.MODE_PREFETCH)
    assert tr.into_proof() == golden


# ------------------------------------------------------------------------------------------------ one proof over several GPUs, device-side exchange
def _emulate_ranks_dev(api, ctx, world, cap_words, prove_shard_dev, emit_shard_dev):
    """The exchange of api.ShardExchange with all `world` ranks emulated on one device: every rank writes its partial buffer into
    its row of the gathered buffer (what the NCCL all-gather produces), one merge kernel, rank 0 serialises."""
    import torch
    gathered = torch.zeros(world * cap_words, dtype=torch.int64, device="cuda")
    merged = torch.zeros(cap_words, dtype=torch.int64, device="cuda")
    n = None
    for r in range(world - 1, -1, -1):        # rank 0 last: its node / circuit keeps the deferred serialisers
        part = torch.zeros(cap_words, dtype=torch.int64, device="cuda")
        nw = prove_shard_dev(r, world, part.data_ptr(), cap_words)
        ctx.synchronize()
        assert n is None or n == nw
        n = nw
        gathered[r * n:(r + 1) * n] = part[:n]
    torch.cuda.synchronize()
    api.shard_merge_device(ctx, gathered.data_ptr(), world, n, merged.data_ptr())
    return emit_shard_dev(merged.data_ptr(), n)


@pytest.mark.parametrize("name,world", [("1024_1x27_65537", 2), ("4096_2x55_65537", 4), ("4096_2x55_65537", 8)])
def test_lasso_node_sharded_device_exchange(api, ctx, oracle, golden_dir, name, world):
    P, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, golden_dir)
    node, pp, tr0, pt0, val0 = _prove_gpu(api, ctx, bounds, segs, nv, inp)
    want = tr0.into_proof()
    tr = api.Keccak256Transcript()
    buf = api.DeviceBuffer.from_numpy(ctx, inp)
    pt, val = _emulate_ranks_dev(api, ctx, world, node.shard_words,
                                 lambda r, w, ptr, cap: node.prove_shard_dev(buf, tr if r == 0 else api.Keccak256Transcript(), r, w, ptr, cap, n_inputs=inp.size),
                                 node.emit_shard_dev)
    assert tr.into_proof() == want and (pt == pt0).all() and (val == val0).all()
    node.free()


@pytest.mark.parametrize("name,world", [("1024_1x27_65537", 2), ("4096_2x55_65537", 3), ("4096_2x55_65537", 8)])
def test_full_gkr_prove_sharded_equals_single_device(api, ctx, golden_dir, name, world):
    """hg_gkr_prove_shard_dev: ONE gkr::prove_gkr (every Vanilla / FFT / product node and the Lasso node) split over `world`
    ranks, all emulated on this device; merged bytes == the single-device proof, input claims identical."""
    from hyper_greco_b200 import params
    P = params.PARAMS[name]
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    d_ct = api.DeviceBuffer.from_numpy(ctx, io["ct0is"])
    want, claims0 = prover.prove(dev, d_ct, 0)
    L = prover.ct0is_log2_size

    def out_claims(tr):
        point = tr.squeeze_challenges(L)
        value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
        return [(np.zeros((0, point.shape[1]), np.uint64), np.zeros(point.shape[1], np.uint64)), (point, value)]

    tr = api.Keccak256Transcript()

    def shard(r, w, ptr, cap):
        t = tr if r == 0 else api.Keccak256Transcript()
        return prover.circuit.prove_gkr_shard_dev(out_claims(t), t, r, w, ptr, cap)

    claims = _emulate_ranks_dev(api, ctx, world, prover.circuit.shard_words, shard, prover.circuit.emit_shard_dev)
    assert tr.into_proof() == want
    assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for ca, cb in zip(claims0, claims) for a, b in zip(ca, cb))
    # the unsharded path still works on the same circuit afterwards
    again, _ = prover.prove(dev, d_ct, 0)
    assert again == want


@pytest.mark.parametrize("name,world", [("1024_1x27_65537", 2), ("4096_2x55_65537", 3), ("4096_2x55_65537", 8)])
def test_full_gkr_prove_sharded_parts_concatenate_to_the_proof(api, ctx, golden_dir, name, world):
    """hg_gkr_emit_shard_part_dev: the serialisation of a sharded proof split over the ranks. Every part is emitted from the merged
    message buffer (here by the one emulated circuit, whose serialisers are those every rank holds); the parts, concatenated in
    order and appended to rank 0's transcript, are the single-device proof, and the input claims are the same after every part."""
    import torch
    from hyper_greco_b200 import params
    P = params.PARAMS[name]
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    d_ct = api.DeviceBuffer.from_numpy(ctx, io["ct0is"])
    want, claims0 = prover.prove(dev, d_ct, 0)
    L = prover.ct0is_log2_size
    tr = api.Keccak256Transcript()
    head = len(tr.into_proof())

    def shard(r, w, ptr, cap):
        t = tr if r == 0 else api.Keccak256Transcript()
        point = t.squeeze_challenges(L)
        value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
        return prover.circuit.prove_gkr_shard_dev([(np.zeros((0, point.shape[1]), np.uint64), np.zeros(point.shape[1], np.uint64)), (point, value)], t, r, w, ptr, cap)

    parts, claims = [], []

    def emit_parts(d_merged, n):
        for p in range(world):
            parts.append(prover.circuit.emit_shard_part_dev(d_merged, n, p, world))
            claims.append(prover.circuit._read_input_claims())
        return None

    _emulate_ranks_dev(api, ctx, world, prover.circuit.shard_words, shard, emit_parts)
    assert head == 0 and all(len(x) > 0 for x in parts)
    for x in parts:
        tr.append_bytes(x)
    assert tr.into_proof() == want
    for cl in claims:
        assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for ca, cb in zip(claims0, cl) for a, b in zip(ca, cb))
    again, _ = prover.prove(dev, d_ct, 0)   # the unsharded path still works on the same circuit afterwards
    assert again == want


def test_full_gkr_prove_sharded_full_size(api, ctx, golden_dir):
    """BASELINE.json config 4 (n=32768 k=16 Goldilocks, one proof over 2/4/8 GPUs): 4 emulated ranks give the committed sha256."""
    from hyper_greco_b200 import params, witness
    meta = _fullsize_meta(golden_dir, "goldilocks_bfv_encrypt_n32768_seed5")
    P = params.by_n(32768)
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, 5))
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs(ins)
    d_ct = api.DeviceBuffer.from_numpy(ctx, np.array(ct0is, dtype=np.uint64))
    prover.circuit.evaluate(dev)
    L = prover.ct0is_log2_size
    tr = api.Keccak256Transcript()

    def shard(r, w, ptr, cap):
        t = tr if r == 0 else api.Keccak256Transcript()
        point = t.squeeze_challenges(L)
        value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
        return prover.circuit.prove_gkr_shard_dev([(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (point, value)], t, r, w, ptr, cap)

    _emulate_ranks_dev(api, ctx, 4, prover.circuit.shard_words, shard, prover.circuit.emit_shard_dev)
    _assert_hash(tr.into_proof(), meta, "sharded BfvEncrypt::prove n=32768, 4 ranks")


# ------------------------------------------------------------------------------------------------ witness generator on the device
@pytest.mark.parametrize("name,seed", [("1024_1x27_65537", 1), ("4096_2x55_65537", 2), ("8192_4x55_65537", 3)])
def test_device_witness_generator_equals_numpy_restatement(api, ctx, name, seed):
    """hg_bfv_witness_generate (scripts/circuit_sk.py:72-140 on the device: exact a_i s over Z, centred reductions, r2i, r1i, bound
    asserts, get_inputs layout) == hyper-greco_b200/witness.py on the same random draws, element for element."""
    from hyper_greco_b200 import params, witness
    P = params.PARAMS[name]
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, seed))
    want = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
    dev, d_ct = witness.synth_witness_device(ctx, P, seed)
    assert len(dev) == len(want)
    for k, (b, w) in enumerate(zip(dev, want)):
        got = b.download(np.uint64, len(w))
        assert (got == np.array(w, dtype=np.uint64)).all(), k
    assert (d_ct.download(np.uint64, len(ct0is)) == np.array(ct0is, dtype=np.uint64)).all()


def test_device_witness_generator_full_size_and_bn254(api, ctx, ctx_bn):
    """n=32768, k=16: the generated witness satisfies the circuit (the `sum` layer of circuit.evaluate equals ct0is,
    sk_encryption_circuit.rs:280-285) and its proof verifies with the product's host verifier; BN254 output equals the numpy
    restatement at n=1024; a witness that violates a bound is refused."""
    from hyper_greco_b200 import params, witness
    P = params.by_n(32768)
    dev, d_ct = witness.synth_witness_device(ctx, P, 7)
    prover = api.BfvSkEncryptProver(ctx, P)
    prover.circuit.evaluate(dev)
    ptr, n = prover.circuit.node_value(prover.ids["sum"])

    class NodeValue:  # library-owned device memory, wrapped for mle_eval_batch
        pass
    nvw = NodeValue()
    nvw.ptr = ptr
    L = prover.ct0is_log2_size
    assert n == 1 << L
    pt = api.Keccak256Transcript().squeeze_challenges(L)
    assert (api.mle_eval_batch(ctx, nvw, 1, L, pt)[0] == api.mle_eval_batch(ctx, d_ct, 1, L, pt)[0]).all()   # sum layer == ct0is (Schwartz-Zippel)
    proof, _ = prover.prove(dev, d_ct, 0)
    ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, 7))
    flat = [np.array(v, dtype=np.uint64) for v in [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]]
    api.BfvSkEncryptVerifier(P).verify(flat, np.array(ct0is, dtype=np.uint64), proof)
    # BN254: canonical limbs after decoding == numpy restatement mod r
    Pn = params.PARAMS["1024_1x27_65537"]
    insb, ctb = witness.get_inputs(Pn, witness.synth_witness(Pn, 4, p=witness.BN_R))
    devb, d_ctb = witness.synth_witness_device(ctx_bn, Pn, 4)
    wantb = [insb["s"], insb["e"], insb["k1"]] + list(insb["ais"]) + list(insb["r1is"]) + [insb["r2is"]]
    for b, w in zip(devb, wantb):
        assert (b.to_field(len(w)) == _bn_limbs(w)).all()
    assert (d_ctb.to_field(len(ctb)) == _bn_limbs(ctb)).all()
    # a bound that the witness violates (r1 bound 0) is an error, as the reference script's assert
    import dataclasses
    bad = dataclasses.replace(Pn, R1_BOUNDS=(0,))
    with pytest.raises(api.HgError):
        witness.synth_witness_device(ctx, bad, 4)


def test_product_event_log_equals_interchange_dump(api, ctx, golden_dir):
    """The order in which the PRODUCT squeezes and writes (interactive schedule, caller-owned transcript) is the order of the committed
    interchange dump (tests/golden/dumps, scripts/hg_dump.py): same S/W pattern, same challenges, same elements. This is the file a
    real run of the Rust prover is diffed against (patches/hyper-greco-dump.diff)."""
    import importlib.util
    from hyper_greco_b200 import params
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("hg_dump", os.path.join(root, "scripts", "hg_dump.py"))
    hd = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(hd)
    name = "1024_1x27_65537"
    _, events = hd.read_dump(os.path.join(hd.DUMP_DIR, f"bfv_encrypt_goldilocks_{name}_{hd.setting_tag(hd.SETTINGS[0])}.hgdump"))
    P = params.PARAMS[name]
    io = np.load(os.path.join(golden_dir, f"circuit_io_{name}.npz"))
    prover = api.BfvSkEncryptProver(ctx, P)
    dev = prover.upload_inputs({k: io[k] for k in ("s", "e", "k1", "ais", "r1is", "r2is")})
    d_ct = api.DeviceBuffer.from_numpy(ctx, io["ct0is"])
    prover.circuit.evaluate(dev)
    tr = api.CallbackTranscript(api.Keccak256Transcript())
    L = prover.ct0is_log2_size
    point = tr.squeeze_challenges(L)
    value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
    prover.circuit.prove_gkr([(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (point, value)], tr, api.MODE_INTERACTIVE)
    got = []
    for kind, limbs in tr.log:            # one extension element = two base-field events of the same kind
        for b in limbs:
            got.append(("S" if kind == "squeeze" else "W", int(b).to_bytes(8, "big")))
    assert got == events


# ------------------------------------------------------------------------------------------------ plug-in lookup types (table.rs:16-67)
def test_plugin_lookup_types_on_the_device(api, ctx, golden_dir):
    """hg_lasso_preprocess_lookups + hg_lasso_node_new_ids: (1) RangeLookup written out as table data proves to the committed golden
    bytes (the plug-in path IS the built-in path); (2) a genuinely different table (16-bit squares, two chunks, weight 3) next to a
    range check: the product's verifier accepts the proof, the claimed sum is sum_k eq(r, k) * (sq[lo] + 3 sq[hi]) resp. the range
    output, and a row that reads outside its lookup's chunk bits is truncated as the reference does (lasso.rs:388-389)."""
    from hyper_greco_b200 import params, witness
    name = "1024_1x27_65537"
    P = params.PARAMS[name]
    golden = open(os.path.join(golden_dir, f"proof_goldilocks_lasso_node_{name}.bin"), "rb").read()
    inp = np.load(os.path.join(golden_dir, f"lasso_inputs_{name}.npz"))["inputs"]
    bounds, segs, nv = witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)
    pp = api.LassoPreprocessing.preprocess_lookups([api.range_lookup_as_table(b) for b in bounds])
    node = api.LassoNode(ctx, pp, nv, [(f"range_{b}", l) for b, l in segs])
    tr = api.Keccak256Transcript()
    node.prove_claim_reduction(inp, tr)
    assert tr.into_proof() == golden
    node.free()
    # (2) custom table
    M = 1 << 16
    sq = np.array([(i * i) & 0xFFFF for i in range(M)], np.uint64)
    pp2 = api.LassoPreprocessing.preprocess_lookups([api.TableLookup("sq16", [("sq", sq, [0, 1])], [16, 16], 3), api.range_lookup_as_table(65537)])
    rng = np.random.default_rng(5)
    n_sq, n_rg, nv2 = 3000, 1000, 12
    x_sq = rng.integers(0, 1 << 32, n_sq, dtype=np.uint64)
    x_sq[0] = (1 << 40) | 0x12345678                                  # bits above the lookup's 32 are dropped
    x_rg = rng.integers(0, 65537, n_rg, dtype=np.uint64)
    inputs = np.concatenate([x_sq, x_rg])
    node2 = api.LassoNode(ctx, pp2, nv2, [("sq16", n_sq), ("range_65537", n_rg)])
    tr2 = api.Keccak256Transcript()
    pt, val = node2.prove_claim_reduction(inputs, tr2)
    proof = tr2.into_proof()
    vpt, vval = api.lasso_node_verify(pp2, nv2, api.Keccak256Transcript(api.GOLDILOCKS, proof))
    assert (vpt == pt).all() and (vval == val).all()
    lo, hi = x_sq & 0xFFFF, (x_sq >> 16) & 0xFFFF
    out = np.zeros(1 << nv2, np.uint64)
    out[:n_sq] = sq[lo] + 3 * sq[hi]
    out[n_sq:n_sq + n_rg] = x_rg                                       # range_65537: full limb + 65536 * remainder limb = the value itself
    assert (api.mle_eval_host(api.GOLDILOCKS, out, nv2, pt) == val).all()
    bad = bytearray(proof)
    bad[-5] ^= 1
    with pytest.raises(api.HgError):
        api.lasso_node_verify(pp2, nv2, api.Keccak256Transcript(api.GOLDILOCKS, bytes(bad)))
    node2.free()

