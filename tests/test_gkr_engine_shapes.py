"""The generic GKR layer engine at every shape where its host-side classifiers, fast paths and round schedule switch.

The device engine (csrc/gkr_dev.cuh, csrc/gkr_kernels.cuh) picks one of several kernels per node: the element-wise product
sumcheck or the general two-phase one, forward evaluation by gate runs (k_vanilla_runs) or per gate (k_vanilla_eval), reverse
wiring by runs (k_wiring_runs) or per element (k_wiring_gather), streamed rounds, the tail kernel and three ways of capturing a
linear layer's input evaluations, and launch grids shaped by every job in the launch. Each circuit of CASES aims at one of these
switches (its comment names the branch); seeded random DAGs draw sizes around the same thresholds.

The reference is the CPU restatement (oracle/ plus tests/general_layer_oracle.cpp), and plain Python integers for the forward
values of small layers and FFTs and for the MLE of small inputs. On the CPU: the restatement evaluates every circuit as the
Python reference does, proves and verifies it, every input claim is the exact MLE of its input at a point of the input's size,
and the library's host verifier accepts the restatement's proof with the same input claims. On the GPU (-m gpu): every node's
device value, the proof bytes and the input claims equal the restatement's in prefetch mode, in interactive mode and with a
callback transcript, and the host verifier accepts the device proof.

A circuit is an op list: ("input", log2_size, num_reps), ("fft", log2_size, inverse), ("vanilla", arity, log2_sub, segments,
num_reps), ("connect", from, to). A layer's gates come in segments (n, const, adds, muls): gate j of the segment has the
constant `const` (None: none), an edge (coef, (inp, (w0 + j step) mod 2^log2_sub)) per add (coef, inp, w0, step), and a
product term per mul (coef, i0, w0, s0, i1, w1, s1) the same way on both sides. A coefficient None is one."""
import ctypes as C
import random

import numpy as np
import pytest

from test_general_layer import FIELDS, GL_P, PRIME, GeneralOracle, _gp, _glib, _gchk, device_values, rand_ext, same_claims

KEYS = ("has_const", "consts", "add_ptr", "add_coef", "add_in", "add_wire", "mul_ptr", "mul_coef", "mul_in0", "mul_w0", "mul_in1", "mul_w1")
PROD_TAIL_LOG = 9  # HG_PROD_TAIL_LOG (gkr_kernels.cuh): the last 9 rounds of a job with nv >= 3 run in the tail kernel
FFT_MAX = {0: 20, 1: 16}  # the largest transform the shared-memory NTT tiles accept (ntt_engine.cuh)


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


# ------------------------------------------------------------------------------------------------ op lists
class Ops(list):
    """an op list with helpers that append a node and its connections and return the node's id"""

    def node(self, op, preds=()):
        nid = sum(1 for o in self if o[0] != "connect")
        self.append(op)
        self.extend(("connect", p, nid) for p in preds)
        return nid

    def input(self, lg, reps=1):
        return self.node(("input", lg, reps))

    def fft(self, src, lg, inverse=False):
        return self.node(("fft", lg, inverse), [src])

    def vanilla(self, preds, log2_sub, segs, reps=1):
        return self.node(("vanilla", len(preds), log2_sub, list(segs), reps), preds)

    def relays(self, src, lg, count):
        """`count` identity layers reading `src` (2^lg entries): `src` gets one claim from each"""
        return [self.vanilla([src], lg, [relay(1 << lg)]) for _ in range(count)]


def relay(n, inp=0, w0=0, step=1, coef=None, const=None):
    return (n, const, [(coef, inp, w0, step)], [])


def emul(n):
    """out[g] = in0[g] in1[g]"""
    return (n, None, [], [(None, 0, 0, 1, 1, 0, 1)])


def node_shapes(ops):
    """(kind, out_len) per node and the output nodes (no successors, not inputs) in insertion order"""
    nodes, succ = [], set()
    for op in ops:
        if op[0] == "input":
            nodes.append(("input", op[2] << op[1]))
        elif op[0] == "fft":
            nodes.append(("fft", 1 << op[1]))
        elif op[0] == "vanilla":
            n = sum(s[0] for s in op[3]) * op[4]
            nodes.append(("vanilla", 1 << (n - 1).bit_length()))
        else:
            succ.add(op[1])
    return nodes, [i for i, (k, _) in enumerate(nodes) if k != "input" and i not in succ]


def layer_csr(segs, log2_sub, field):
    """segments -> the CSR arrays of hg_circuit_insert_vanilla (field elements as limbs [n, LIMBS])"""
    from oracle import hgo
    sub, k, p = 1 << log2_sub, hgo.LIMBS[field], PRIME[field]
    felts = lambda vals: hgo.ints_to_limbs([(1 if v is None else int(v)) % p for v in vals], field).reshape(-1, k)
    out = {key: [] for key in KEYS}
    n_add, n_mul = [], []
    for n, const, adds, muls in segs:
        j = np.arange(n, dtype=np.int64)[:, None]
        wires = lambda w0, st: ((np.array(w0, np.int64)[None, :] + j * np.array(st, np.int64)[None, :]) % sub).reshape(-1).astype(np.uint64)
        out["has_const"].append(np.full(n, const is not None, np.uint8))
        out["consts"].append(np.repeat(felts([0 if const is None else const]), n, axis=0))
        n_add.append(np.full(n, len(adds), np.uint64))
        n_mul.append(np.full(n, len(muls), np.uint64))
        if adds:
            out["add_coef"].append(np.tile(felts([a[0] for a in adds]), (n, 1)))
            out["add_in"].append(np.tile(np.array([a[1] for a in adds], np.uint32), n))
            out["add_wire"].append(wires([a[2] for a in adds], [a[3] for a in adds]))
        if muls:
            out["mul_coef"].append(np.tile(felts([m[0] for m in muls]), (n, 1)))
            out["mul_in0"].append(np.tile(np.array([m[1] for m in muls], np.uint32), n))
            out["mul_w0"].append(wires([m[2] for m in muls], [m[3] for m in muls]))
            out["mul_in1"].append(np.tile(np.array([m[4] for m in muls], np.uint32), n))
            out["mul_w1"].append(wires([m[5] for m in muls], [m[6] for m in muls]))
    dt = {"has_const": np.uint8, "add_in": np.uint32, "mul_in0": np.uint32, "mul_in1": np.uint32}
    res = {}
    for key in KEYS:
        if key.endswith("_ptr"):
            continue
        empty = np.zeros((0, k) if key in ("consts", "add_coef", "mul_coef") else 0, dt.get(key, np.uint64))
        res[key] = np.ascontiguousarray(np.concatenate(out[key] or [empty]))
    res["add_ptr"] = np.concatenate([np.zeros(1, np.uint64), np.cumsum(np.concatenate(n_add), dtype=np.uint64)])
    res["mul_ptr"] = np.concatenate([np.zeros(1, np.uint64), np.cumsum(np.concatenate(n_mul), dtype=np.uint64)])
    return res


class Restatement(GeneralOracle):
    """GeneralOracle with layers inserted from segments (CSR arrays straight into hgt_insert_vanilla)"""

    def insert_vanilla(self, arity, log2_sub, segs, num_reps=1):
        a = layer_csr(segs, log2_sub, self.field)
        i = C.c_int(-1)
        _gchk(_glib().hgt_insert_vanilla(self.h, arity, log2_sub, num_reps, len(a["has_const"]), *[_gp(a[k]) for k in KEYS], C.byref(i)))
        return i.value


def build(builder, ops, field):
    """the circuit on the restatement or on the library (device circuit, or host description for verify_gkr)"""
    ids = []
    for op in ops:
        if op[0] == "input":
            ids.append(builder.insert_input(op[1], op[2]))
        elif op[0] == "fft":
            ids.append(builder.insert_fft(op[1], op[2]))
        elif op[0] == "vanilla":
            if isinstance(builder, Restatement):
                ids.append(builder.insert_vanilla(op[1], op[2], op[3], op[4]))
            else:
                a = layer_csr(op[3], op[2], field)
                ids.append(builder.insert_vanilla_arrays(op[1], op[2], op[4], *[a[k] for k in KEYS]))
        else:
            builder.connect(op[1], op[2])
    return ids


def random_limbs(field, rng, n):
    """n nonzero canonical base elements as limbs (BN254: the top limb below 2^61 keeps the value below r)"""
    if field == 0:
        return rng.integers(1, GL_P, size=n, dtype=np.uint64)
    v = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64)
    v[:, 0] |= np.uint64(1)
    v[:, 3] >>= np.uint64(2)
    return v.reshape(-1)


def instance(hgo, ops, field, seed=0):
    """-> (restatement circuit evaluated on random inputs, inputs, output claims at random points)"""
    rng = np.random.default_rng(seed)
    nodes, outs = node_shapes(ops)
    oc = Restatement(field)
    build(oc, ops, field)
    ins = [random_limbs(field, rng, n) for kind, n in nodes if kind == "input"]
    oc.evaluate(ins)
    claims = []
    for o in outs:
        nv = (nodes[o][1] - 1).bit_length()
        pt = rand_ext(field, rng, nv)
        claims.append((pt, hgo.mle_eval(field, oc.value(o), nv, pt)))
    return oc, ins, claims


# ------------------------------------------------------------------------------------------------ plain Python reference
PY_MAX = 1 << 13  # forward values and MLEs in Python integers up to this many entries


def ints(hgo, limbs, field):
    return hgo.limbs_to_ints(limbs, field)


def ext_int(row, field):
    """an extension element [el] limbs -> (c0, c1) of F[X] / (X^2 - 7) (BN254: degree one, c1 = 0)"""
    row = [int(x) for x in np.asarray(row).reshape(-1)]
    return (row[0], row[1]) if field == 0 else (sum(x << (64 * i) for i, x in enumerate(row)), 0)


def py_mle(table, point, p):
    """MLE of a base table at an extension point, lowest variable first"""
    assert len(table) == 1 << len(point)
    t = [(x, 0) for x in table]
    for r0, r1 in point:
        t = [(a0 + r0 * (b0 - a0) + 7 * r1 * (b1 - a1), a1 + r0 * (b1 - a1) + r1 * (b0 - a0)) for (a0, a1), (b0, b1) in zip(t[::2], t[1::2])]
        t = [(x % p, y % p) for x, y in t]
    return t[0]


def py_layer(op, xs, p):
    """forward values of a Vanilla layer from its segments; xs: the input slots' values"""
    _, _, log2_sub, segs, reps = op
    sub = 1 << log2_sub
    out = []
    for r in range(reps):
        for n, const, adds, muls in segs:
            for j in range(n):
                v = 0 if const is None else const
                for c, i, w0, st in adds:
                    v += (1 if c is None else c) * xs[i][r * sub + (w0 + j * st) % sub]
                for c, i0, w0, s0, i1, w1, s1 in muls:
                    v += (1 if c is None else c) * xs[i0][r * sub + (w0 + j * s0) % sub] * xs[i1][r * sub + (w1 + j * s1) % sub]
                out.append(v % p)
    return out + [0] * ((1 << (len(out) - 1).bit_length()) - len(out))


def py_dft(hgo, x, field, inverse):
    """naive DFT with the field's primitive root of order len(x): out[k] = sum_j x_j w^(jk) (inverse: w^-1, scaled by 1/n)"""
    p, n = PRIME[field], len(x)
    lg = n.bit_length() - 1
    delta = hgo.ints_to_limbs([0, 1] + [0] * (n - 2), field)
    w = ints(hgo, hgo.ntt(field, delta, lg), field)[1]  # the transform of the delta at 1 is the powers of the root
    assert pow(w, n, p) == 1 and (n == 1 or pow(w, n // 2, p) == p - 1)
    if inverse:
        w = pow(w, p - 2, p)
    out = [sum(x[j] * pow(w, j * k, p) for j in range(n)) % p for k in range(n)]
    return [v * pow(n, p - 2, p) % p for v in out] if inverse else out


def check_forward(hgo, ops, field, value):
    """every small layer and FFT recomputed in Python integers from its inputs' values; value(i) -> limbs of node i"""
    nodes, _ = node_shapes(ops)
    preds = {}
    for op in ops:
        if op[0] == "connect":
            preds.setdefault(op[2], []).append(op[1])
    ops_nodes = [op for op in ops if op[0] != "connect"]
    checked = 0
    for i, op in enumerate(ops_nodes):
        if op[0] == "vanilla" and nodes[i][1] <= PY_MAX and all(nodes[q][1] <= PY_MAX for q in preds[i]) and len(set(preds[i])) <= 64:
            cache = {q: ints(hgo, value(q), field) for q in set(preds[i])}
            assert ints(hgo, value(i), field) == py_layer(op, [cache[q] for q in preds[i]], PRIME[field]), f"node {i}: forward value"
            checked += 1
        elif op[0] == "fft" and nodes[i][1] <= 64:
            assert ints(hgo, value(i), field) == py_dft(hgo, ints(hgo, value(preds[i][0]), field), field, op[2]), f"node {i}: FFT value"
            checked += 1
    return checked


def check_input_claims(hgo, ops, field, ins, claims):
    """every claim on an input is the MLE of that input at a point of the input's size"""
    nodes, _ = node_shapes(ops)
    sizes = [n for kind, n in nodes if kind == "input"]
    assert len(claims) == len(ins)
    for vec, n, cl in zip(ins, sizes, claims):
        tab = ints(hgo, vec, field) if n <= PY_MAX else None
        for pt, v in cl:
            assert pt.shape[0] == (n - 1).bit_length(), "claim point shorter or longer than its input"
            if tab is not None and pt.shape[0] <= 12:
                assert py_mle(tab, [ext_int(r, field) for r in pt], PRIME[field]) == ext_int(v, field)
            else:
                assert (hgo.mle_eval(field, vec, pt.shape[0], pt) == v).all()


def host_verify(api, ops, field, claims, proof):
    c = api.Circuit(None, field)
    build(c, ops, field)
    return c.verify_gkr(claims, api.Keccak256Transcript.from_proof(proof, field))


# ------------------------------------------------------------------------------------------------ circuits
# Every case is a function of the field returning an op list; its comment names the branch of the engine it targets.
def em_case(ng, log2_sub=3, reps=1):
    def f(field):
        o = Ops()
        a, b = o.input(log2_sub, reps), o.input(log2_sub, reps)
        o.vanilla([a, b], log2_sub, [emul(ng)], reps)
        return o
    return f


def lin_case(arity, log2_sub, segs, reps=1, claims=1):
    """one linear layer over `arity` inputs of reps << log2_sub entries, with `claims` claims"""
    def f(field):
        o = Ops()
        ins = [o.input(log2_sub, reps) for _ in range(arity)]
        lay = o.vanilla(ins, log2_sub, segs, reps)
        if claims > 1:
            n = node_shapes(o)[0][lay][1]
            o.relays(lay, (n - 1).bit_length(), claims)
        return o
    return f


def slot_gates(arity, log2_sub):
    """one gate per input slot k: (k + 2) X_k[k mod 2^log2_sub], so every slot is read"""
    return [(1, None, [(k + 2, k, k % (1 << log2_sub), 0)], []) for k in range(arity)]


def schedule_case(nv):
    """Round schedule at nv = log2 S: element-wise products and linear layers with m = log2(n_in) at 1, stream_end - 1,
    stream_end, stream_end + 1, nv - 1 and nv (where the arity stays within 4096), arity 1 (read in place) and arity > 1 with
    a_pad != arity, and one, two and three claims. m < stream_end: captured by the copy after streamed round m; stream_end <= m
    < nv: captured in the tail at cap_round = m - stream_end; m == nv: the last fold. nv < 3 has no tail."""
    se = nv if nv < 3 else max(2, nv - PROD_TAIL_LOG)
    ms = sorted({m for m in (1, se - 1, se, se + 1, nv - 1, nv) if 1 <= m <= nv and nv - m <= 12})

    def f(field):
        o = Ops()
        a, b = o.input(nv), o.input(nv)
        em = o.vanilla([a, b], nv, [emul(1 << nv)])
        o.relays(em, nv, 0 if nv >= 20 else 1 + nv % 3)   # 1 / 2 / 3 claims (an output node has one)
        for q, m in enumerate(ms):
            k = nv - m
            arity = 1 if k == 0 else (2 if k == 1 else (1 << (k - 1)) + 1)
            x = o.input(m)
            extra = [relay(min(1 << m, 64), inp=arity - 1, w0=1, step=1, coef=5, const=(3 if q % 2 else None))]
            lay = o.vanilla([x] * arity, m, slot_gates(arity, m) + extra)
            n = node_shapes(o)[0][lay][1]
            o.relays(lay, (n - 1).bit_length(), q % 3 + 1 if q % 3 else 0)
        return o
    return f


def shaping_case(big):
    """Launch shaping: linear layers (reversed wiring: one wiring run per element, k_wiring_runs), linear layers that read every
    element twice (k_wiring_gather), element-wise products and FFTs of 2^1 .. 2^12 entries,
    with (big) or without a 2^20-entry linear layer in the same round launches. round_pairs sums over every job of a launch,
    so the small nodes are reduced with different pairs per thread and block counts in the two circuits. With `big` the circuit
    also holds FFT nodes of log2_size 1 and of the largest size the field's NTT tiles accept."""
    def f(field):
        o = Ops()
        for lg in range(1, 13):
            x, y = o.input(lg), o.input(lg)
            o.vanilla([x], lg, [relay(1 << lg, w0=(1 << lg) - 1, step=-1, coef=lg + 1)])
            o.vanilla([y], lg, [(1 << lg, None, [(lg + 1, 0, (1 << lg) - 1, -1), (2, 0, 0, 1)], [])])
            o.vanilla([x, y], lg, [emul(1 << lg)])
        if big:
            z = o.input(20)
            o.vanilla([z], 20, [relay(1 << 20, coef=3, const=1)])
            f1 = o.fft(o.input(1), 1)
            o.fft(f1, 1, inverse=True)
            top = FFT_MAX[field]
            o.fft(o.input(top), top)
        return o
    return f


def run_break(kind):
    """16 relays X[g] in one forward run and one wiring run, broken at gate 7 by one wire, one coefficient or one constant"""
    w = {"wire": (12, None, None), "coef": (7, 9, None), "const": (7, None, 4)}[kind]
    return [relay(7), (1, w[2], [(w[1], 0, w[0], 0)], []), relay(8, w0=8)]


def runs_case(n_runs, reps):
    """n_runs forward runs per rep (gate g reads wire 2g: no two gates extend one run); fwd_runs * num_reps > 4096 takes the
    per-gate kernel"""
    def f(field):
        lg = (2 * n_runs - 1).bit_length()
        o = Ops()
        x = o.input(lg, reps)
        o.vanilla([x], lg, [relay(n_runs, step=2, coef=7)], reps)
        return o
    return f


def wire_runs_case(extra_run):
    """2048 gates reading wires 0, 2, .., 4094 of 4096: 4096 alternating copy and zero wiring runs (k_wiring_runs). With
    `extra_run` the input has 8192 elements and one more gate reads the last one: elements 4095 .. 8190 make one zero run and
    element 8191 a 4097th run, one over the limit (k_wiring_gather)"""
    def f(field):
        lg = 13 if extra_run else 12
        o = Ops()
        x = o.input(lg)
        o.vanilla([x], lg, [relay(2048, step=2)] + ([relay(1, w0=8191, step=0)] if extra_run else []))
        return o
    return f


def fwd_edges_case(ne):
    """gates with ne additive edges over three inputs (HG_FWD_MAXE = 5: 5 edges take the run kernel, 6 the per-gate one)"""
    adds = [(i + 2, i % 3, i, 1) for i in range(ne)]
    return lin_case(3, 4, [(16, 11, adds, [])])


def input_alignment_case(field):
    """Inputs of 1 and 2 entries before an 8-entry one that a relay and an FFT read in place with 32-byte vector loads: the
    inputs are packed into one device arena, where each must start 32-byte aligned (a misaligned address fault otherwise)"""
    o = Ops()
    o.input(0)
    o.input(1)
    x = o.input(3)
    o.vanilla([x], 3, [relay(8, coef=3)])
    o.fft(x, 3)
    return o


def general_repeated_case(field):
    """A general layer that reads one layer in slots 0 and 1 and one input in slots 2 and 3: each of those nodes gets the
    phase-1 and phase-2 claims of one slot before those of the next, in the order the verifier reads them"""
    o = Ops()
    x, y = o.input(3), o.input(3)
    lay = o.vanilla([x], 3, [relay(8, coef=2)])
    o.vanilla([lay, lay, y, y], 3, [(8, 1, [(3, 2, 0, 1)], [(None, 0, 0, 1, 1, 7, -1), (5, 2, 1, 1, 3, 0, 1)])])
    return o


CASES = {
    # item 1: element-wise product classification. 8 gates over 8 wires: the element-wise product sumcheck. 4 (a smaller power
    # of two), 5 and 7 gates leave wires unread and 4 gates over 2 reps repeat: all of them the general two-phase layer sumcheck
    "em_full": em_case(8),
    "em_pow2_short": em_case(4),
    "em_5_gates": em_case(5),
    "em_7_gates": em_case(7),
    "em_reps2": em_case(4, log2_sub=2, reps=2),
    # item 2: forward runs (k_vanilla_runs) against k_vanilla_eval
    "fwd_5_edges": fwd_edges_case(5),
    "fwd_6_edges": fwd_edges_case(6),
    "fwd_break_wire": lin_case(1, 4, run_break("wire")),
    "fwd_break_coef": lin_case(1, 4, run_break("coef")),
    "fwd_break_const": lin_case(1, 4, run_break("const")),
    # constant-only gates (ne == 0) before, between and after relays; the zero padding to out_len (21 gates -> 32)
    "fwd_const_only": lin_case(2, 4, [(3, 5, [], []), relay(8, inp=1), (2, 0, [], []), relay(8, coef=3, const=2)]),
    "fwd_runs_4096": runs_case(4096, 1),
    "fwd_runs_4097": runs_case(4097, 1),
    "fwd_runs_2048_reps2": runs_case(2048, 2),
    "fwd_runs_2049_reps2": runs_case(2049, 2),
    # n_gates num_reps = 10, not a power of two: padding after the last rep
    "fwd_pad_reps2": lin_case(2, 3, [relay(2, w0=3), (1, 9, [(2, 1, 0, 0), (3, 0, 7, 0)], []), relay(2, inp=1, step=3)], reps=2),
    # item 3: reverse wiring runs (k_wiring_runs kinds zero / copy / scaled) against k_wiring_gather
    "wire_identity": lin_case(1, 5, [relay(32)]),
    "wire_scaled": lin_case(1, 5, [relay(32, coef=GL_P - 1)]),
    "wire_mixed": lin_case(1, 5, [relay(8), relay(8, w0=8, coef=3), relay(8, w0=16, coef=4), relay(8, w0=24)]),
    "wire_read_twice": lin_case(1, 4, [relay(8), relay(1, w0=3, step=0, coef=2), relay(7, w0=8)]),
    "wire_gaps": lin_case(2, 5, [relay(5, w0=2), relay(6, w0=11, coef=6), relay(4, inp=1, w0=20, step=2)]),
    "wire_arity3": lin_case(3, 3, [relay(8), relay(8, inp=1, coef=2), relay(8, inp=2, w0=0)]),
    "wire_runs_4096": wire_runs_case(False),
    "wire_runs_4097": wire_runs_case(True),
    # the order of the claims a general layer puts on a node that fills several of its slots
    "general_repeated_input": general_repeated_case,
    # the layout of the inputs on the device
    "input_alignment": input_alignment_case,
    # item 4: round schedule
    **{f"schedule_nv{nv}": schedule_case(nv) for nv in (1, 2, 3, 10, 11, 12, 13, 20)},
    # item 5: launch shaping (and FFT sizes)
    "shaping_alone": shaping_case(False),
    "shaping_with_2p20": shaping_case(True),
}


# ------------------------------------------------------------------------------------------------ random circuits
LOG_SIZES = (1, 2, 3, 9, 10, 11, 12, 13)


def random_ops(seed):
    """a random DAG of inputs, FFTs, linear, element-wise and general layers with sizes around the engine's thresholds"""
    rng = random.Random(seed)
    o = Ops()
    sizes = []  # log2 out_len per node

    def around(lg):  # a gate count at, just below or just above 2^lg
        return max(1, (1 << lg) + rng.choice((0, 0, -1, 1)))

    def coef():
        return rng.choice((None, None, 1, 2, GL_P - 1, rng.randrange(1, 2**62)))

    for _ in range(rng.randint(1, 3)):
        lg = rng.choice(LOG_SIZES)
        reps = 2 if lg > 1 and rng.random() < 0.3 else 1
        o.input(lg - (reps == 2), reps)
        sizes.append(lg)
    for _ in range(rng.randint(3, 6)):
        kind = rng.choice(("linear", "linear", "emul", "general", "fft"))
        src = rng.randrange(len(sizes))
        lg = sizes[src]
        same = [i for i, s in enumerate(sizes) if s == lg]
        if kind == "fft":
            o.fft(src, lg, rng.random() < 0.5)
            sizes.append(lg)
            continue
        reps = 2 if lg > 1 and rng.random() < 0.25 else 1
        sub_lg = lg - (reps == 2)
        sub = 1 << sub_lg
        if kind == "emul":
            ng = sub if rng.random() < 0.6 else rng.randint(1, sub)
            nid = o.vanilla([src, rng.choice(same)], sub_lg, [emul(ng)], reps)
        else:
            arity = rng.randint(1, 3)
            segs, left = [], around(rng.choice((1, 3, 9, 10, 12))) if kind == "linear" else rng.randint(1, 40)
            while left > 0:
                n = min(left, rng.choice((1, 2, 7, 64, 1 << 12)))
                left -= n
                const = None if rng.random() < 0.6 else rng.randrange(0, 2**62)
                ne = rng.choice((0, 1, 1, 1, 2, 5, 6)) if kind == "linear" else rng.randint(0, 2)
                adds = [(coef(), rng.randrange(arity), rng.randrange(sub), rng.choice((0, 1, 1, 1, 2, -1))) for _ in range(ne)]
                muls = [] if kind == "linear" else [(coef(), rng.randrange(arity), rng.randrange(sub), rng.choice((0, 1, 3)),
                                                     rng.randrange(arity), rng.randrange(sub), rng.choice((0, 1, 2))) for _ in range(rng.randint(1, 2))]
                segs.append((n, const, adds, muls))
            nid = o.vanilla([rng.choice(same) for _ in range(arity)], sub_lg, segs, reps)
        sizes.append((node_shapes(o)[0][nid][1] - 1).bit_length())
    return o


SEEDS = list(range(20))


# ------------------------------------------------------------------------------------------------ CPU
def check_restatement(api, hgo, ops, field, seed=0):
    oc, ins, claims = instance(hgo, ops, field, seed)
    check_forward(hgo, ops, field, oc.value)
    proof, pclaims = oc.prove_gkr(claims)
    assert same_claims(oc.verify_gkr(claims, proof), pclaims)
    check_input_claims(hgo, ops, field, ins, pclaims)
    assert same_claims(host_verify(api, ops, field, claims, proof), pclaims)


def printed_on_failure(name, ops, fn):
    try:
        fn()
    except BaseException:
        print(f"op list of {name}:\n{list(ops)!r}")
        raise


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("field", FIELDS)
def test_restatement_proves_and_host_verifier_accepts(api, hgo, field, case):
    ops = CASES[case](field)
    check_restatement(api, hgo, ops, field)


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("field", FIELDS)
def test_random_circuit_restatement(api, hgo, field, seed):
    ops = random_ops(seed)
    printed_on_failure(f"random seed {seed}", ops, lambda: check_restatement(api, hgo, ops, field, seed))


@pytest.mark.parametrize("ng", [4, 5, 7])
@pytest.mark.parametrize("field", FIELDS)
def test_partial_elementwise_product_is_a_general_layer(api, hgo, field, ng):
    """gates out[g] = in0[g] in1[g] for g < ng over 8-entry inputs whose other wires are nonzero: the restatement's proof verifies,
    the host verifier accepts it, and every input claim is the input's MLE at a point of 3 variables (the input's size). Proved by
    the element-wise product sumcheck over pad2(ng) entries, the unread wires would be missing from the sum, and the claims would
    have log2 pad2(ng) variables."""
    ops = em_case(ng)(field)
    oc, ins, claims = instance(hgo, ops, field, seed=ng)
    proof, pclaims = oc.prove_gkr(claims)
    assert same_claims(oc.verify_gkr(claims, proof), pclaims)
    assert same_claims(host_verify(api, ops, field, claims, proof), pclaims)
    for vec, cl in zip(ins, pclaims):
        assert len(cl) == 2  # the general layer's two phases each put one claim on every input
        for pt, v in cl:
            assert pt.shape[0] == 3
            assert py_mle(ints(hgo, vec, field), [ext_int(r, field) for r in pt], PRIME[field]) == ext_int(v, field)


@pytest.mark.parametrize("field", FIELDS)
def test_num_reps_not_a_power_of_two_is_refused(api, field):
    """num_reps 3 would give an input of 3 << log2_size entries, or a layer reading such inputs: tables the sumchecks cannot fold.
    The library (device and host circuits share the rule) and the restatement refuse them when they are inserted."""
    c = api.Circuit(None, field)
    with pytest.raises(api.HgError, match="power of two"):
        c.insert_input(3, 3)
    c.insert_input(3, 2)
    a = layer_csr([relay(4)], 3, field)
    with pytest.raises(api.HgError, match="power of two"):
        c.insert_vanilla_arrays(1, 3, 3, *[a[k] for k in KEYS])
    assert c.insert_vanilla_arrays(1, 3, 2, *[a[k] for k in KEYS]) == 1
    r = Restatement(field)
    with pytest.raises(Exception, match="power of two"):
        r.insert_input(3, 3)
    with pytest.raises(Exception, match="power of two"):
        r.insert_vanilla(1, 3, [relay(4)], 3)


def planned_runs(op, field=0):
    """The device's run planning for one linear layer (GkrCircuitDev::insert_vanilla), restated: (forward runs, wiring runs),
    each a count, or None where the planner falls back to the per-gate / per-element kernel"""
    _, arity, log2_sub, segs, reps = op
    a = layer_csr(segs, log2_sub, field)
    ng, sub = len(a["has_const"]), 1 << log2_sub
    n_in, a_pad = reps << log2_sub, 1 << (arity - 1).bit_length()
    ptr, ins, wires = [int(x) for x in a["add_ptr"]], [int(x) for x in a["add_in"]], [int(x) for x in a["add_wire"]]
    coefs = [tuple(int(v) for v in row) for row in a["add_coef"]]
    consts = [tuple(int(v) for v in row) if h else (0,) * row.size for h, row in zip(a["has_const"], a["consts"])]
    fwd = []  # [g0, len, edges [(input, first wire, coefficient)], constant]
    for g in range(ng):
        edges = [(ins[e], wires[e], coefs[e]) for e in range(ptr[g], ptr[g + 1])]
        if len(edges) > 5:
            fwd = None
            break
        last = fwd[-1] if fwd else None
        if last and len(last[2]) == len(edges) and last[3] == consts[g] and all(
                i == li and w == lw + g - last[0] and c == lc for (i, w, c), (li, lw, lc) in zip(edges, last[2])):
            last[1] += 1
            continue
        fwd.append([g, 1, edges, consts[g]])
        if len(fwd) * reps > 4096:
            fwd = None
            break
    readers = {}
    for r in range(reps):
        for g in range(ng):
            for e in range(ptr[g], ptr[g + 1]):
                readers.setdefault(ins[e] * n_in + r * sub + wires[e], []).append((r * ng + g, coefs[e]))
    runs = []  # [kind, out0, len, coefficient]
    for x in range(a_pad * n_in):
        rd = readers.get(x, [])
        if len(rd) > 1:
            return (None if fwd is None else len(fwd)), None
        last = runs[-1] if runs else None
        if not rd:
            if last and last[0] == 0:
                last[2] += 1
            else:
                runs.append([0, 0, 1, None])
        else:
            o, c = rd[0]
            if last and last[0] != 0 and last[1] + last[2] == o and last[3] == c:
                last[2] += 1
            else:
                runs.append([1, o, 1, c])
        if len(runs) > 4096:
            return (None if fwd is None else len(fwd)), None
    return (None if fwd is None else len(fwd)), len(runs)


# (forward runs, wiring runs) of the first layer of each run case, None = the fallback kernel: keeps every case on its branch
RUN_BRANCHES = {
    "fwd_5_edges": (5, None), "fwd_6_edges": (None, None), "fwd_break_wire": (3, None), "fwd_break_coef": (3, 3),
    "fwd_break_const": (3, 1), "fwd_const_only": (4, 4), "fwd_runs_4096": (4096, None), "fwd_runs_4097": (None, None),
    "fwd_runs_2048_reps2": (2048, None), "fwd_runs_2049_reps2": (None, None), "fwd_pad_reps2": (4, None),
    "wire_identity": (1, 1), "wire_scaled": (1, 1), "wire_mixed": (4, 4), "wire_read_twice": (3, None), "wire_gaps": (6, 13),
    "wire_arity3": (3, 4), "wire_runs_4096": (2048, 4096), "wire_runs_4097": (2049, None),
}


@pytest.mark.parametrize("case", list(RUN_BRANCHES))
def test_run_cases_take_their_branch(case):
    op = next(op for op in CASES[case](0) if op[0] == "vanilla")
    assert planned_runs(op) == RUN_BRANCHES[case]


def test_random_ops_are_reproducible():
    """a failing seed's op list is the circuit that seed builds, so it can be pasted into CASES"""
    assert random_ops(3) == random_ops(3) and random_ops(3) != random_ops(4)
    assert any(op[0] == "vanilla" for s in SEEDS for op in random_ops(s))


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


def check_device(api, hgo, ctx, ops, field, seed=0):
    oc, ins, claims = instance(hgo, ops, field, seed)
    want, wclaims = oc.prove_gkr(claims)
    c = api.Circuit(ctx)
    ids = build(c, ops, field)
    c.evaluate_host(ins)
    for i in ids:
        assert (device_values(api, ctx, c, i) == oc.value(i)).all(), f"node {i}: device value"
    for mode in (api.MODE_PREFETCH, api.MODE_INTERACTIVE):
        tr = api.Keccak256Transcript(field)
        got = c.prove_gkr(claims, tr, mode)
        assert tr.into_proof() == want, f"mode {mode}: proof bytes"
        assert same_claims(got, wclaims), f"mode {mode}: input claims"
    tr = api.CallbackTranscript(api.Keccak256Transcript(field), field)
    got = c.prove_gkr(claims, tr, api.MODE_PREFETCH)
    proof = tr.into_proof()
    assert proof == want and same_claims(got, wclaims), "callback transcript"
    assert same_claims(host_verify(api, ops, field, claims, proof), got)
    check_input_claims(hgo, ops, field, ins, got)
    c.free()


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("field", FIELDS)
def test_device_matches_restatement(api, hgo, ctxs, field, case):
    check_device(api, hgo, ctxs(field), CASES[case](field), field)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("field", FIELDS)
def test_random_circuit_device(api, hgo, ctxs, field, seed):
    ops = random_ops(seed)
    printed_on_failure(f"random seed {seed}", ops, lambda: check_device(api, hgo, ctxs(field), ops, field, seed))


@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_device_circuit_refusals(api, hgo, ctxs, field):
    """a device circuit refuses num_reps 3 on an input and on a layer, and an input pointer that is not 32-byte aligned, before
    it launches anything; the same circuit then evaluates from an aligned pointer"""
    ctx = ctxs(field)
    c = api.Circuit(ctx)
    with pytest.raises(api.HgError, match="power of two"):
        c.insert_input(3, 3)
    x = c.insert_input(3)
    a = layer_csr([relay(8, coef=3)], 3, field)
    with pytest.raises(api.HgError, match="power of two"):
        c.insert_vanilla_arrays(1, 3, 3, *[a[k] for k in KEYS])
    lay = c.insert_vanilla_arrays(1, 3, 1, *[a[k] for k in KEYS])
    c.connect(x, lay)
    vals = random_limbs(field, np.random.default_rng(1), 8)
    buf = api.DeviceBuffer.from_field(ctx, np.concatenate([vals, vals]).reshape(16, -1) if field else np.concatenate([vals, vals]))

    class At:  # a device pointer as Circuit.evaluate takes it
        def __init__(self, ptr):
            self.ptr = ptr
    with pytest.raises(api.HgError, match="32-byte aligned"):
        c.evaluate([At(buf.ptr + 8)])
    c.evaluate([At(buf.ptr)])
    want = hgo.ints_to_limbs([3 * v % PRIME[field] for v in ints(hgo, vals, field)], field)
    assert (device_values(api, ctx, c, lay) == want).all()
    c.free()
    buf.free()
