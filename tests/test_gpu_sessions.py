"""Proofs made the way a proving service makes them: many live objects of different shapes in one context, several contexts of one
field, one context per host thread (bench.py's in-flight slots), contexts on several devices. Every proof is checked against an
exact reference: the committed golden bytes, the committed full-size sha256, the CPU oracle, or the CPU restatement of general
layers (tests/test_general_layer.py).

The kernels that take dynamic shared memory share one limit per kernel and device across the whole process
(cudaFuncAttributeMaxDynamicSharedMemorySize). A CPU test checks that every such kernel gets its limit in the one place that sets
them, at context creation, so no object's shapes can lower the limit another object's launches need."""
import hashlib
import json
import os
import re
import threading

import numpy as np
import pytest

from conftest import load_case
from test_general_layer import build, make_instance, same_claims

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CSRC = os.path.join(ROOT, "hyper-greco_b200", "csrc")
GL_P = 2**64 - 2**32 + 1
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
N1024 = "1024_1x27_65537"
TAG = {0: "goldilocks", 1: "bn254"}


# ------------------------------------------------------------------------------------------------ CPU: one place sets the limits
def _strip_comments(src):
    return re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)


def _csrc():
    return {f: _strip_comments(open(os.path.join(CSRC, f)).read()) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".hpp"))}


KERNEL_DEF = re.compile(r"__global__\s+void\s+(?:__launch_bounds__\s*\([^)]*\)\s*)?(\w+)\s*\(")
LAUNCH = re.compile(r"(\w+)\s*(?:<[^<>;]*(?:<[^<>;]*>[^<>;]*)*>)?\s*<<<(.*?)>>>", re.S)


def _split_args(s):
    """top-level comma split of a launch configuration"""
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "([{<":
            depth += 1
        elif ch in ")]}>":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    return out + [cur.strip()]


def _dynamic_smem_kernels(sources):
    """kernels that declare extern __shared__ memory, and kernels launched with a dynamic shared-memory size other than 0"""
    found = {}
    for f, src in sources.items():
        defs = [(m.start(), m.group(1)) for m in KERNEL_DEF.finditer(src)]
        for m in re.finditer(r"extern\s+__shared__", src):
            owner = [name for pos, name in defs if pos < m.start()]
            assert owner, f"{f}: extern __shared__ outside a kernel"
            found.setdefault(owner[-1], f"{f}: extern __shared__")
        for m in LAUNCH.finditer(src):
            args = _split_args(m.group(2))
            if len(args) >= 3 and args[2] != "0":
                found.setdefault(m.group(1), f"{f}: launched with {args[2]} bytes")
    return found


def _limits_function(sources):
    src = sources["abi.cu"]
    m = re.search(r"void\s+set_dynamic_smem_limits\s*\([^)]*\)\s*\{", src)
    assert m, "abi.cu: set_dynamic_smem_limits is missing"
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(src[i], 0)
        i += 1
    return src[m.start():i]


def test_one_place_sets_every_dynamic_shared_memory_limit():
    sources = _csrc()
    kernels = _dynamic_smem_kernels(sources)
    # the scan finds the kernels it is meant to find
    assert {"k_ntt_cols", "k_ntt_rows", "k_prod_tail", "k_prod_tail_one", "k_prod_mid_one", "k_gp_tail", "k_tree_tail"} <= set(kernels)
    body = _limits_function(sources)
    for k, where in kernels.items():
        assert re.search(r"\b" + k + r"\s*<\s*FP\s*>", body), f"{k} ({where}) takes dynamic shared memory, but set_dynamic_smem_limits does not set its limit"
    sets = {f: src.count("cudaFuncAttributeMaxDynamicSharedMemorySize") for f, src in sources.items()}
    assert body.count("cudaFuncAttributeMaxDynamicSharedMemorySize") == 1
    assert sum(sets.values()) == 1, f"the dynamic shared-memory limit is also set outside set_dynamic_smem_limits: {sets}"
    # and both fields get their limits when a context is created
    create = re.search(r"int\s+hg_ctx_create\s*\(.*?\n\}", sources["abi.cu"], re.S).group(0)
    for fp in ("GlField", "FrField"):
        assert re.search(r"set_dynamic_smem_limits\s*<\s*" + fp + r"\s*>", create), fp


# ------------------------------------------------------------------------------------------------ GPU: objects and their references
@pytest.fixture(scope="module")
def api():
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api
    api.lib()  # raises if the CUDA library is missing: no fallback
    return api


def _golden(fname):
    return open(os.path.join(GOLDEN, fname), "rb").read()


def _fullsize(key):
    meta = json.load(open(os.path.join(GOLDEN, "golden_proofs.json"))).get("fullsize", {})
    if key not in meta:
        pytest.skip(f"{key} not generated yet (tests/golden/make_golden_fullsize.py)")
    return meta[key]


def _matches_hash(meta):
    return lambda proof: len(proof) == meta["bytes"] and hashlib.sha256(proof).hexdigest() == meta["sha256"]


def _bn_limbs(vals):
    return np.array([[(int(v) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for v in vals], dtype=np.uint64)


_WITNESS = {}


def _bfv_witness(field, n, seed):
    """host vectors (get_inputs order) and ct0is of the synthetic witness, as limbs of `field`"""
    key = (field, n, seed)
    if key not in _WITNESS:
        from hyper_greco_b200 import params, witness
        P = params.by_n(n)
        if field == 0:
            ins, ct = witness.get_inputs(P, witness.synth_witness(P, seed))
            conv = lambda v: np.array(v, dtype=np.uint64).reshape(-1)
        else:
            ins, ct = witness.get_inputs(P, witness.synth_witness(P, seed, p=witness.BN_R))
            conv = lambda v: _bn_limbs(v).reshape(-1)
        flat = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
        _WITNESS[key] = (P, [conv(v) for v in flat], conv(ct))
    return _WITNESS[key]


class Obj:
    """One live object of a session: run() proves once with it and returns what its caller receives, check(out) compares that
    with the object's reference."""

    def __init__(self, label, run, check, owned):
        self.label, self.run, self.check, self.owned = label, run, check, owned

    def use(self):
        assert self.check(self.run()), self.label

    def free(self):
        for o in self.owned:
            o.free()


def bfv_golden(api, ctx):
    from hyper_greco_b200 import params
    tag = TAG[ctx.field]
    io = np.load(os.path.join(GOLDEN, f"circuit_io_{N1024}.npz" if ctx.field == 0 else f"circuit_io_bn254_{N1024}.npz"))
    flat = [np.ascontiguousarray(v).reshape(-1) for v in [io["s"], io["e"], io["k1"]] + list(io["ais"]) + list(io["r1is"]) + [io["r2is"]]]
    ct = np.ascontiguousarray(io["ct0is"]).reshape(-1)
    want = _golden(f"proof_{tag}_bfv_encrypt_{N1024}.bin")
    prover = api.BfvSkEncryptProver(ctx, params.PARAMS[N1024])
    return Obj(f"{tag} BfvEncrypt n=1024", lambda: prover.prove_host(flat, ct)[0], lambda got: got == want, [prover.circuit, prover.lasso])


def bfv_fullsize(api, ctx, n, seed):
    meta = _fullsize(f"{TAG[ctx.field]}_bfv_encrypt_n{n}_seed{seed}")
    P, flat, ct = _bfv_witness(ctx.field, n, seed)
    prover = api.BfvSkEncryptProver(ctx, P)
    return Obj(f"{TAG[ctx.field]} BfvEncrypt n={n} seed {seed}", lambda: prover.prove_host(flat, ct)[0], _matches_hash(meta), [prover.circuit, prover.lasso])


def _lasso_node(api, ctx, P):
    from hyper_greco_b200 import witness
    pp = api.LassoPreprocessing.preprocess(witness.lasso_lookup_bounds(P))
    return api.LassoNode(ctx, pp, witness.lasso_num_vars(P), witness.lasso_lookup_segments(P))


def _lasso_run(api, node, inp):
    def run():
        tr = api.Keccak256Transcript(node.ctx.field)
        pt, val = node.prove_claim_reduction(inp, tr)
        return tr.into_proof(), pt, val
    return run


def lasso_golden(api, ctx):
    from hyper_greco_b200 import params
    tag = TAG[ctx.field]
    inp = np.load(os.path.join(GOLDEN, f"lasso_inputs_{N1024}.npz" if ctx.field == 0 else f"lasso_inputs_bn254_{N1024}.npz"))["inputs"]
    want = _golden(f"proof_{tag}_lasso_node_{N1024}.bin")
    node = _lasso_node(api, ctx, params.PARAMS[N1024])
    return Obj(f"{tag} Lasso node n=1024", _lasso_run(api, node, inp), lambda got: got[0] == want, [node])


def lasso_oracle(api, ctx, oracle, name):
    P, inp, bounds, segs, nv, opp, rows = load_case(name, oracle, GOLDEN)
    oproof, orr, osum, _ = oracle.lasso_prove(0, opp, nv, rows, inp)
    node = _lasso_node(api, ctx, P)
    check = lambda got: got[0] == oproof and (got[1].reshape(-1) == orr).all() and (got[2] == osum).all()
    return Obj(f"Lasso node {name}", _lasso_run(api, node, inp), check, [node])


def lasso_fullsize(api, ctx):
    from hyper_greco_b200 import params, witness
    meta = _fullsize(f"{TAG[ctx.field]}_lasso_node_n32768_seed0")
    P = params.by_n(32768)
    if ctx.field == 0:
        inp = np.array(witness.lasso_inputs(P, witness.synth_witness(P, 0)), dtype=np.uint64)
    else:
        inp = _bn_limbs(witness.lasso_inputs(P, witness.synth_witness(P, 0, p=witness.BN_R), p=witness.BN_R))
    node = _lasso_node(api, ctx, P)
    match = _matches_hash(meta)
    return Obj(f"{TAG[ctx.field]} Lasso node n=32768", _lasso_run(api, node, inp), lambda got: match(got[0]), [node])


def general_circuit(api, ctx, hgo, case):
    ops, oc, ins, claims = make_instance(hgo, api, ctx.field, case)
    want, wclaims = oc.prove_gkr(claims)
    c = api.Circuit(ctx)
    build(c, ops)

    def run():
        c.evaluate_host(ins)
        tr = api.Keccak256Transcript(ctx.field)
        got = c.prove_gkr(claims, tr, api.MODE_PREFETCH)
        return tr.into_proof(), got
    return Obj(f"{TAG[ctx.field]} {case} circuit", run, lambda got: got[0] == want and same_claims(got[1], wclaims), [c])


def ntt_job(api, ctx, oracle, log_n, batch=2):
    rng = np.random.default_rng(100 + log_n)
    if ctx.field == 0:
        x = rng.integers(0, GL_P, size=(batch, 1 << log_n), dtype=np.uint64)
    else:
        x = rng.integers(0, 2**64, size=(batch, 1 << log_n, 4), dtype=np.uint64)
        x[..., 3] %= np.uint64(BN_R >> 192)
    want = oracle.ntt(ctx.field, x, log_n, False).reshape(x.shape)

    def run():
        if ctx.field == 0:
            d = api.DeviceBuffer.from_numpy(ctx, x)
            api.ntt(ctx, d, log_n, False, batch)
            got = d.download(np.uint64, x.size).reshape(x.shape)
        else:
            d = api.DeviceBuffer.from_field(ctx, x)
            api.ntt(ctx, d, log_n, False, batch)
            got = d.to_field(batch << log_n).reshape(x.shape)
        d.free()
        return got
    return Obj(f"{TAG[ctx.field]} NTT log_n={log_n}", run, lambda got: (got == want).all(), [])


def plugin_node(api, ctx):
    """A plug-in Lasso node with 32 memories: four lookups of one subtable each, every subtable serving all 8 chunks. Its
    grand-product tail kernel needs more than 48 KB of shared memory. The host verifier accepts its proof, the claim is the MLE of
    the combined operands sum_d w^d T[chunk_d(x)], and every later proof has the bytes of the first.

    As in the reference (range.rs:254-256, lasso_host.hpp), chunk_bits only sets how many low bits of an input a lookup reads;
    those bits are then split into uniform log2(M)-bit chunks, chunk d being bits [16 d, 16 d + 16). With 62 bits, chunks 0..3
    carry the input, chunks 4..7 read entry 0, and bit 62 and above are dropped."""
    M, log2M, C_, nv = 1 << 16, 16, 8, 10
    chunk_bits = [16, 16, 16, 10, 1, 1, 1, 1]
    total = sum(chunk_bits)
    rng = np.random.default_rng(29)
    tables = [rng.integers(0, 1 << 32, M, dtype=np.uint64) for _ in range(4)]
    weights = [3, 5, 7, (1 << 20) + 7]
    lookups = [api.TableLookup(f"t{s}", [(f"s{s}", tables[s], list(range(C_)))], chunk_bits, weights[s]) for s in range(4)]
    pp = api.LassoPreprocessing.preprocess_lookups(lookups, C_=C_, M=M)
    assert pp.num_memories == 32
    rows = (1 << nv) // 4
    x = rng.integers(0, 1 << 63, 1 << nv, dtype=np.uint64)
    out = np.zeros(1 << nv, np.uint64)
    for s in range(4):
        for i in range(s * rows, (s + 1) * rows):
            v = int(x[i]) & ((1 << total) - 1)
            out[i] = sum(pow(weights[s], d, GL_P) * int(tables[s][(v >> (log2M * d)) & (M - 1)]) for d in range(C_)) % GL_P
    node = api.LassoNode(ctx, pp, nv, [(f"t{s}", rows) for s in range(4)])
    first = []

    def check(got):
        proof, pt, val = got
        vpt, vval = api.lasso_node_verify(pp, nv, api.Keccak256Transcript(api.GOLDILOCKS, proof))
        assert (vpt == pt).all() and (vval == val).all(), "the host verifier's claim differs from the prover's"
        assert (api.mle_eval_host(api.GOLDILOCKS, out, nv, pt) == val).all(), "the claim is not the MLE of the combined operands"
        if not first:
            first.append(proof)
        return proof == first[0]
    return Obj("plug-in Lasso node, 32 memories", _lasso_run(api, node, x), check, [node])


# ------------------------------------------------------------------------------------------------ GPU: many objects per context
def _session_objects(api, oracle, hgo, ctx, field):
    """every object of one field, in the order they are built and first used. Larger shared-memory requirements of a kernel come
    before smaller ones (k_gp_tail by memory count, k_prod_tail: BfvEncrypt before the small general layers, the NTTs by size),
    so every object is used again after an object with a smaller requirement has been built and used."""
    if field == 0:
        makers = [lambda: plugin_node(api, ctx), lambda: lasso_fullsize(api, ctx), lambda: bfv_fullsize(api, ctx, 32768, 5),
                  lambda: bfv_fullsize(api, ctx, 16384, 3), lambda: lasso_oracle(api, ctx, oracle, "4096_2x55_65537"),
                  lambda: lasso_golden(api, ctx), lambda: bfv_golden(api, ctx), lambda: general_circuit(api, ctx, hgo, "mixed"),
                  lambda: general_circuit(api, ctx, hgo, "random")] + [lambda k=k: ntt_job(api, ctx, oracle, k) for k in (16, 11, 3)]
    else:
        makers = [lambda: lasso_fullsize(api, ctx), lambda: bfv_fullsize(api, ctx, 32768, 5), lambda: lasso_golden(api, ctx),
                  lambda: bfv_golden(api, ctx), lambda: general_circuit(api, ctx, hgo, "mixed")] + \
                 [lambda k=k: ntt_job(api, ctx, oracle, k) for k in (16, 3)]
    objs = []
    try:
        for make in makers:
            objs.append(make())
    except BaseException:
        for o in objs:
            o.free()
        raise
    return objs


@pytest.mark.gpu
@pytest.mark.parametrize("field", [pytest.param(0, id="goldilocks"), pytest.param(1, id="bn254")])
def test_interleaved_objects_keep_their_bytes(api, oracle, field):
    """All objects of one field live in one context, and a small Lasso node lives in a second context of the same field. Every
    object is built first; then each proves in forward order and again in reverse order, with the second context's node proving
    after every one of them."""
    from oracle import hgo
    ctx, ctx2 = api.Context(0, field), api.Context(0, field)
    objs, other = [], None
    try:
        objs = _session_objects(api, oracle, hgo, ctx, field)
        other = lasso_golden(api, ctx2)
        for o in objs + objs[::-1]:
            o.use()
            other.use()
    finally:
        for o in objs + ([other] if other else []):
            o.free()
        ctx.close()
        ctx2.close()


# ------------------------------------------------------------------------------------------------ GPU: one context per thread
def _run_threads(workers):
    errs = []

    def wrap(f):
        def go():
            try:
                f()
            except BaseException as e:  # re-raised in the main thread after join
                errs.append(e)
        return go
    ths = [threading.Thread(target=wrap(f)) for f in workers]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:  # the failure itself, not the broken barrier it left the other threads
        raise next((e for e in errs if not isinstance(e, threading.BrokenBarrierError)), errs[0])


@pytest.mark.gpu
def test_concurrent_contexts_match_the_references(api, oracle):
    """bench.py's conditions: one Context per host thread, the C calls run concurrently. Four threads with different workloads build
    their objects on their own thread and prove 3 times each; one of them first makes a call that is rejected, and afterwards its
    hg_last_error is its own message while the others' is empty. Then bench.py's own setup: 4 slots of BfvEncrypt n=32768 on the
    same witness, prove_gkr on device-resident values in prefetch mode, 3 proofs per slot. Every result is checked after join."""
    from oracle import hgo
    from hyper_greco_b200 import params
    for key in (0, 32768, 5), (0, 16384, 3):  # host witnesses are prepared before the threads start
        _bfv_witness(*key)
    bn_lasso = np.load(os.path.join(GOLDEN, f"lasso_inputs_bn254_{N1024}.npz"))["inputs"]
    workloads = {
        "gl n=32768": (0, lambda ctx: [bfv_fullsize(api, ctx, 32768, 5)]),
        "gl n=16384": (0, lambda ctx: [bfv_fullsize(api, ctx, 16384, 3)]),
        "bn254 n=1024": (1, lambda ctx: [bfv_golden(api, ctx), lasso_golden(api, ctx)]),
        "gl n=1024 + circuit + NTT": (0, lambda ctx: [bfv_golden(api, ctx), general_circuit(api, ctx, hgo, "mixed")] +
                                      [ntt_job(api, ctx, oracle, k) for k in (16, 11, 3)]),
    }
    rejecting = "bn254 n=1024"
    barrier = threading.Barrier(len(workloads))
    sessions = {}

    def worker(name, field, make):
        def f():
            s = sessions[name] = {"ctx": api.Context(0, field), "objs": []}
            try:
                s["objs"] = make(s["ctx"])
                if name == rejecting:   # a BN254 node with a Goldilocks transcript: rejected before any work
                    with pytest.raises(api.HgError, match="belongs to another field"):
                        s["objs"][1].owned[0].prove_claim_reduction(bn_lasso, api.Keccak256Transcript(api.GOLDILOCKS))
                barrier.wait(timeout=900)  # every thread reads its error text after the rejection, while the others prove
            except BaseException:
                barrier.abort()
                raise
            s["outs"] = [[o.run() for o in s["objs"]] for _ in range(3)]
            s["error"] = api.lib().hg_last_error().decode()
        return f

    try:
        _run_threads([worker(name, field, make) for name, (field, make) in workloads.items()])
        for name, s in sessions.items():
            for k, outs in enumerate(s["outs"]):
                for o, out in zip(s["objs"], outs):
                    assert o.check(out), (name, o.label, k)
        assert "belongs to another field" in sessions[rejecting]["error"]
        assert all(s["error"] == "" for name, s in sessions.items() if name != rejecting), {n: s["error"] for n, s in sessions.items()}
    finally:
        for s in sessions.values():
            for o in s["objs"]:
                o.free()
            s["ctx"].close()

    # bench.py's slots: built one after the other on this thread, then driven from one thread each
    meta = _fullsize("goldilocks_bfv_encrypt_n32768_seed5")
    P, flat, ct = _bfv_witness(0, 32768, 5)
    slots = []
    try:
        for _ in range(4):
            ctx = api.Context(0, api.GOLDILOCKS)
            prover = api.BfvSkEncryptProver(ctx, P)
            dev = [api.DeviceBuffer.from_field(ctx, v) for v in flat]
            d_ct = api.DeviceBuffer.from_field(ctx, ct)
            prover.circuit.evaluate(dev)
            L = prover.ct0is_log2_size
            point = api.Keccak256Transcript().squeeze_challenges(L)
            value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
            claims = [(np.zeros((0, 2), np.uint64), np.zeros(2, np.uint64)), (point, value)]
            slots.append((ctx, prover, dev + [d_ct], claims, []))

        def resident(slot):
            ctx, prover, _, claims, proofs = slot

            def f():
                for _ in range(3):
                    tr = api.Keccak256Transcript()
                    tr.squeeze_challenges(prover.ct0is_log2_size)
                    prover.circuit.prove_gkr(claims, tr, api.MODE_PREFETCH)
                    proofs.append(tr.into_proof())
            return f
        _run_threads([resident(s) for s in slots])
        match = _matches_hash(meta)
        for k, s in enumerate(slots):
            assert len(s[4]) == 3 and all(match(p) for p in s[4]), k
    finally:
        for ctx, prover, bufs, _, _ in slots:
            for b in bufs:
                b.free()
            prover.circuit.free()
            prover.lasso.free()
            ctx.close()


# ------------------------------------------------------------------------------------------------ GPU: two devices, one process
@pytest.mark.gpu
def test_two_devices_in_one_process(api):
    """Contexts on devices 0 and 1 in one process, each with a Lasso node and a BfvEncrypt n=1024 prover, used alternately: every
    proof has the committed golden bytes."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctxs = [api.Context(d, api.GOLDILOCKS) for d in (0, 1)]
    objs = []
    try:
        for c in ctxs:
            objs += [lasso_golden(api, c), bfv_golden(api, c)]
        for _ in range(2):
            for o in objs:
                o.use()
    finally:
        for o in objs:
            o.free()
        for c in ctxs:
            c.close()
