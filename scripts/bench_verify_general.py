"""Verification cost of one general Vanilla layer: the host verifier against the batched device verifier (GkrBatchVerifier).

For S = 2^20 .. 2^22 it builds the general layer of scripts/bench_general_layer.py (arity 2, num_reps 16, Goldilocks), proves it on
cuda:0 in prefetch mode and prints one JSON line per size with
  * the host verifier for one proof (verify_gkr plus the input-claim check, one thread) and the host core it ran on;
  * the batched device verifier at B = 1, 8, 64 with proofs of the library's transcript (the same points, so the weights, A(u),
    the constant part and M(u, v) are computed once per batch; every proof has its own copy of the inputs on the device):
    proofs/s and hg_verifier_timing split into replay / device stages / closing;
  * one batch of proofs with their own points (an absorbing caller transcript), where nothing is shared.
The GPU's name and power limit are read (nvidia-smi, read-only) in the same run.

    python scripts/bench_verify_general.py [--sizes 20,21,22] [--batches 1,8,64] [--per-proof 8] [--reps 5]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import hyper_greco_b200  # noqa: E402,F401
from hyper_greco_b200 import api  # noqa: E402
from bench_general_layer import layer_arrays  # noqa: E402

GL_P = api.GL_P
REPS = 16


class Absorbing:
    """a caller transcript whose squeeze hashes everything written or read so far: every proof gets its own points"""

    def __init__(self, seed, proof=None):
        self.state, self.out, self.proof, self.pos = hashlib.sha256(b"seed%d" % seed).digest(), [], proof, 0

    def squeeze_challenge(self):
        self.state = hashlib.sha256(self.state + b"squeeze").digest()
        return np.array([int.from_bytes(self.state[8 * i: 8 * i + 8], "little") % GL_P for i in range(2)], np.uint64)

    def write_felt_ext(self, v):
        v = np.asarray(v, np.uint64)
        self.out.append(v.copy())
        self.state = hashlib.sha256(self.state + v.tobytes()).digest()

    def read_felt_ext(self):
        v = self.proof[self.pos: self.pos + 2]
        self.pos += 2
        self.state = hashlib.sha256(self.state + v.tobytes()).digest()
        return v

    def into_proof(self):
        return np.concatenate(self.out)


def host_core():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"model": model, "threads_used": 1, "cpus_available": len(os.sched_getaffinity(0))}


def measure(ctx, lg, batches, n_per_proof, reps):
    arrays = layer_arrays(lg, REPS, True, seed=lg)
    log2_sub = arrays[1]
    n_in = REPS << log2_sub
    rng = np.random.default_rng(1)
    ins = [rng.integers(0, GL_P, size=n_in, dtype=np.uint64) for _ in range(2)]

    def circuit(c):
        a, b = c.insert_input(log2_sub, REPS), c.insert_input(log2_sub, REPS)
        g = c.insert_vanilla_arrays(*arrays)
        c.connect(a, g)
        c.connect(b, g)
        return g
    c, h = api.Circuit(ctx), api.Circuit(None, api.GOLDILOCKS)
    g = circuit(c)
    circuit(h)
    d_ins = [api.DeviceBuffer.from_numpy(ctx, x) for x in ins]
    c.evaluate(d_ins)
    ptr, n = c.node_value(g)
    out_buf = api.DeviceBuffer.from_numpy(ctx, api.NodeValueView(ctx, ptr, n).download(np.uint64, n))
    nv = (n - 1).bit_length()

    def claim(pt):
        return [(pt, api.mle_eval_batch(ctx, out_buf, 1, nv, pt)[0])]
    claims = claim(rng.integers(0, GL_P, size=(nv, 2), dtype=np.uint64))
    tr = api.Keccak256Transcript()
    c.prove_gkr(claims, tr, api.MODE_PREFETCH)
    proof = tr.into_proof()
    row = {"log2_S": lg, "num_reps": REPS, "proof_bytes": len(proof)}

    # host verifier: verify_gkr + the input-claim check
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        got = h.verify_gkr(claims, api.Keccak256Transcript.from_proof(proof))
        ok = all((api.mle_eval_host(0, vec, p.shape[0], p) == x).all() for vec, cl in zip(ins, got) for p, x in cl)
        ts.append(time.perf_counter() - t0)
        assert ok
    row["host_ms_per_proof"] = round(1e3 * min(ts), 3)
    row["host_core"] = host_core()

    bv = api.GkrBatchVerifier(ctx, h, max(max(batches), n_per_proof))
    copies = [d_ins] + [[api.DeviceBuffer.from_numpy(ctx, x) for x in ins] for _ in range(max(batches) - 1)]

    def timed(make_trs, oc, inputs):
        best = None
        for i in range(reps + 1):  # the first call sizes the pools
            trs = make_trs()
            t0 = time.perf_counter()
            res = bv.verify_batch(trs, oc, inputs)
            t = time.perf_counter() - t0
            assert all(ok for ok, _ in res), res[0]
            if i and (best is None or t < best[0]):
                best = (t, bv.timing())
        B = len(inputs)
        t, tm = best
        return {"batch": B, "proofs_per_s": round(B / t, 2), "ms_per_batch": round(1e3 * t, 3),
                "replay_ms_per_proof": round(tm["replay_us"] / 1e3 / B, 4), "device_ms": round(tm["device_us"] / 1e3, 3),
                "close_ms": round(tm["close_us"] / 1e3, 4)}
    row["shared_points"] = [timed(lambda: [api.Keccak256Transcript.from_proof(proof) for _ in range(B)], [claims] * B, copies[:B]) for B in batches]

    # proofs with their own points: an absorbing transcript squeezes the output point, then the proof is made interactively
    own = []
    for s in range(n_per_proof):
        inner = Absorbing(s)
        t = api.CallbackTranscript(inner)
        cl = claim(t.squeeze_challenges(nv))
        c.prove_gkr(cl, t, api.MODE_INTERACTIVE)
        own.append((s, cl, inner.into_proof()))

    def own_trs():
        trs = []
        for s, _, pr in own:
            t = api.CallbackTranscript(Absorbing(s, pr))
            t.squeeze_challenges(nv)
            trs.append(t)
        return trs
    row["per_proof_points"] = timed(own_trs, [cl for _, cl, _ in own], [copies[i % len(copies)] for i in range(n_per_proof)])
    bv.free()
    c.free()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20,21,22")
    ap.add_argument("--batches", default="1,8,64")
    ap.add_argument("--per-proof", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    name, power = ([x.strip() for x in gpu.splitlines()[0].split(",")] + ["unknown"])[:2] if gpu.strip() else ("unknown", "unknown")
    ctx = api.Context(0)
    for lg in (int(x) for x in a.sizes.split(",")):
        row = measure(ctx, lg, [int(b) for b in a.batches.split(",")], a.per_proof, a.reps)
        row.update(gpu=name, power_limit=power)
        print(json.dumps(row), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
