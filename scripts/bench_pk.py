"""BFV public-key encryption next to secret-key encryption on one GPU.

For each parameter set and each relation (sk: BfvSkEncryptProver, pk: BfvPkEncryptProver), with a device-generated witness, Goldilocks,
prefetch mode, it prints one JSON line with
  * witness_ms: the device witness generator (hg_bfv_witness_generate / hg_bfv_pk_witness_generate), host draws excluded, best of reps;
  * single_ms: one proof at a time (evaluate + output claims + prove_gkr + serialisation), median over --proofs;
  * proofs_per_s_inflight: --inflight independent proofs resident on the device (one context and one host thread each), --proofs
    proofs per thread;
  * class_ms: per kernel class, device ms of one proof from hg_ctx_profile (median over 3 individually profiled proofs);
  * lasso_node_device_bytes: hg_lasso_node_device_bytes of the Lasso node;
  * verify_batch: batched device verifier proofs/s at B = 1 / 8 / 64 (the same proof and device inputs B times: the points are shared);
  * the GPU's name and power limit, read (nvidia-smi, read-only) in the same run.

    python scripts/bench_pk.py [--sets 4096_2x55_65537,32768_16x59_65537] [--proofs 20] [--inflight 4] [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import hyper_greco_b200  # noqa: E402,F401
from hyper_greco_b200 import api, params, witness  # noqa: E402


class Case:
    """one prover with its device witness on its own context"""

    def __init__(self, kind, name, seed, device=0):
        self.kind, self.ctx = kind, api.Context(device)
        if kind == "sk":
            self.P = params.PARAMS[name]
            self.gen = lambda: witness.synth_witness_device(self.ctx, self.P, seed)
            self.prover = api.BfvSkEncryptProver(self.ctx, self.P)
            self.verifier = api.BfvSkEncryptVerifier(self.P)
        else:
            self.P = params.PK_PARAMS[name]
            self.gen = lambda: witness.synth_pk_witness_device(self.ctx, self.P, seed)
            self.prover = api.BfvPkEncryptProver(self.ctx, self.P)
            self.verifier = api.BfvPkEncryptVerifier(self.P)
        self.w = self.gen()

    def prove(self):
        if self.kind == "sk":
            dev, d_ct = self.w
            return self.prover.prove(dev, d_ct)[0]
        dev, d0, d1 = self.w
        return self.prover.prove(dev, d0, d1)[0]

    def verify_batch(self, proof, B):
        if self.kind == "sk":
            dev, d_ct = self.w
            return self.verifier.verify_batch(self.ctx, [dev] * B, [d_ct] * B, [proof] * B)
        dev, d0, d1 = self.w
        return self.verifier.verify_batch(self.ctx, [dev] * B, [d0] * B, [d1] * B, [proof] * B)

    def close(self):
        b = getattr(self.verifier, "_batch", None)
        if b is not None:
            b.free()
        self.prover.circuit.free()
        self.prover.lasso.free()
        self.w = None
        self.ctx.close()


def measure(kind, name, a):
    c = Case(kind, name, 1)
    row = {"relation": kind, "set": name, "field": "goldilocks", "mode": "prefetch"}
    ts = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        c.w = c.gen()           # synchronises on the device status before it returns
        ts.append(time.perf_counter() - t0)
    row["witness_ms"] = round(1e3 * min(ts), 3)
    proof = c.prove()
    for _ in range(3):
        c.prove()
    ts = []
    for _ in range(a.proofs):
        t0 = time.perf_counter()
        c.prove()
        ts.append(time.perf_counter() - t0)
    row["single_ms"] = round(1e3 * statistics.median(ts), 3)
    row["proof_bytes"] = len(proof)
    runs = []
    for _ in range(3):
        c.ctx.profile(True)
        c.prove()
        runs.append(c.ctx.profile_read())
        c.ctx.profile(False)
    row["class_ms"] = {k: round(statistics.median(r[k][1] for r in runs), 4) for k in runs[0] if any(r[k][0] for r in runs)}
    row["lasso_node_device_bytes"] = c.prover.lasso.device_bytes
    row["lasso_num_vars"] = c.prover.lasso.num_vars
    vb = []
    for B in (1, 8, 64):
        assert all(ok for ok, _ in c.verify_batch(proof, B))
        best = None
        for _ in range(a.reps):
            t0 = time.perf_counter()
            c.verify_batch(proof, B)
            t = time.perf_counter() - t0
            best = t if best is None else min(best, t)
        vb.append({"batch": B, "proofs_per_s": round(B / best, 2)})
    row["verify_batch"] = vb
    c.close()
    # resident throughput: independent proofs in flight, one context and one host thread each
    cases = [Case(kind, name, 1 + k) for k in range(a.inflight)]
    for s in cases:
        s.prove()
    start = threading.Barrier(a.inflight + 1)

    def work(s):
        start.wait()
        for _ in range(a.proofs):
            s.prove()
    ths = [threading.Thread(target=work, args=(s,)) for s in cases]
    for t in ths:
        t.start()
    start.wait()
    t0 = time.perf_counter()
    for t in ths:
        t.join()
    row["proofs_per_s_inflight"] = round(a.inflight * a.proofs / (time.perf_counter() - t0), 2)
    row["inflight"] = a.inflight
    for s in cases:
        s.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="4096_2x55_65537,32768_16x59_65537")
    ap.add_argument("--proofs", type=int, default=20)
    ap.add_argument("--inflight", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    name, power = ([x.strip() for x in gpu.splitlines()[0].split(",")] + ["unknown"])[:2] if gpu.strip() else ("unknown", "unknown")
    for s in a.sets.split(","):
        for kind in ("sk", "pk"):
            row = measure(kind, s, a)
            row.update(gpu=name, power_limit=power)
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
