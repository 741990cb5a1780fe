"""Device cost of one general Vanilla layer (the two-phase layer sumcheck, DESIGN.md section 3) against a linear layer of the same size.

For S = 2^20 .. 2^22 entries of concatenated inputs (arity 2, num_reps 16, one gate per input element and rep, random wiring) it
builds two one-layer circuits on cuda:0: the general one (per gate one product of two random wires with a random coefficient, one
add and a constant on every fourth gate) and the linear one (the same gates without their product). It prints one JSON line per
size: the prove time of each (prefetch mode, host clock around prove_gkr, which ends in a device synchronise) and, from
hg_ctx_profile, the device ms and algorithmic bytes of the layer-weights class (eq tables, wiring, the G / M_u gathers and H(u)) and
of the layer-sumcheck class (both phases for the general layer). The general layer's extra weights time is the cost of the new
kernels. Usage: python scripts/bench_general_layer.py [--sizes 20,21,22] [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hyper_greco_b200  # noqa: E402,F401
from hyper_greco_b200 import api  # noqa: E402

GL_P = 2**64 - 2**32 + 1


def layer_arrays(log2_S, reps, general, seed):
    rng = np.random.default_rng(seed)
    n_in = 1 << (log2_S - 1)                      # arity 2
    log2_sub = (n_in // reps).bit_length() - 1
    sub = 1 << log2_sub
    ng = sub                                      # out_len = ng * reps = n_in
    e = lambda: rng.integers(0, GL_P, size=ng, dtype=np.uint64)
    has_const = (np.arange(ng) % 4 == 0).astype(np.uint8)
    add_ptr = np.arange(ng + 1, dtype=np.uint64)
    mul_ptr = np.arange(ng + 1, dtype=np.uint64) if general else np.zeros(ng + 1, np.uint64)
    nm = ng if general else 0
    return (2, log2_sub, reps, has_const, e(), add_ptr, e(), rng.integers(0, 2, size=ng).astype(np.uint32),
            rng.integers(0, sub, size=ng).astype(np.uint64), mul_ptr, e()[:nm], rng.integers(0, 2, size=nm).astype(np.uint32),
            rng.integers(0, sub, size=nm).astype(np.uint64), rng.integers(0, 2, size=nm).astype(np.uint32), rng.integers(0, sub, size=nm).astype(np.uint64))


def measure(ctx, log2_S, general, iters, reps=16):
    arrays = layer_arrays(log2_S, reps, general, seed=log2_S)
    n_in = 1 << (log2_S - 1)
    rng = np.random.default_rng(1)
    ins = [rng.integers(0, GL_P, size=n_in, dtype=np.uint64) for _ in range(2)]
    c = api.Circuit(ctx)
    a, b = c.insert_input(arrays[1], reps), c.insert_input(arrays[1], reps)
    g = c.insert_vanilla_arrays(*arrays)
    c.connect(a, g)
    c.connect(b, g)
    d_ins = [api.DeviceBuffer.from_numpy(ctx, x) for x in ins]
    c.evaluate(d_ins)
    nv = (n_in - 1).bit_length()
    pt = rng.integers(0, GL_P, size=(nv, 2), dtype=np.uint64)
    ptr, n = c.node_value(g)
    out_buf = api.DeviceBuffer.from_numpy(ctx, api.NodeValueView(ctx, ptr, n).download(np.uint64, n))
    claims = [(pt, api.mle_eval_batch(ctx, out_buf, 1, nv, pt)[0])]

    def prove():
        tr = api.Keccak256Transcript()
        c.prove_gkr(claims, tr, api.MODE_PREFETCH)
        return tr.into_proof()
    for _ in range(3):
        prove()
    ctx.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        prove()
    ms = (time.perf_counter() - t0) / iters * 1e3
    ctx.profile(True)
    for _ in range(3):
        prove()
    prof = ctx.profile_read()
    ctx.profile(False)
    cls = {k: {"launches": v[0] / 3, "ms": round(v[1] / 3, 4), "bytes": int(v[2] / 3)} for k, v in prof.items() if k.startswith("gkr_layer")}
    c.free()
    return {"prove_ms": round(ms, 4), "classes": cls}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20,21,22")
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip()
    ctx = api.Context(0)
    for lg in (int(x) for x in args.sizes.split(",")):
        row = {"log2_S": lg, "gpu": gpu.splitlines()[0] if gpu else "unknown"}
        row["general"] = measure(ctx, lg, True, args.iters)
        row["linear"] = measure(ctx, lg, False, args.iters)
        print(json.dumps(row), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
