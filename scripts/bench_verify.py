"""Proofs/s of the batched device verifier (BfvSkEncryptVerifier.verify_batch) against the host verifier (verify), one JSON line
per configuration. Batches of B copies of one device-made proof of a synthetic witness (every proof of the library's transcript
carries the same points, so the weights are shared), each proof with its own copy of the inputs, resident on the device or as host
vectors. Also the host replay time per proof and the per-class device time and bytes of a batch.

    python scripts/bench_verify.py [--n 32768] [--fields 0,1] [--batches 1,8,64,256] [--reps 3]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hyper_greco_b200  # noqa: E402,F401
from hyper_greco_b200 import api, params, witness  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=32768)
    ap.add_argument("--fields", default="0,1")
    ap.add_argument("--batches", default="1,8,64,256")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    P = params.by_n(a.n)
    for field in [int(f) for f in a.fields.split(",")]:
        ctx = api.Context(0, field)
        limbs = api.LIMBS[field]
        ins, ct0is = witness.get_inputs(P, witness.synth_witness(P, 1, api.GL_P if field == 0 else api.BN_R))
        vals = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
        to_limbs = (lambda v: np.array(v, dtype=np.uint64).reshape(-1)) if limbs == 1 else \
            (lambda v: np.array([[(int(x) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for x in v], np.uint64).reshape(-1))
        flat = [to_limbs(v) for v in vals]
        ct = to_limbs(ct0is)
        prover = api.BfvSkEncryptProver(ctx, P)
        proof, _ = prover.prove_host(flat, ct, 0)
        ver = api.BfvSkEncryptVerifier(P, field)
        t0 = time.perf_counter()
        ver.verify(flat, ct, proof)
        host_s = time.perf_counter() - t0
        def upload():  # one proof's inputs and ct0is on the device, in the library's representation
            bufs = [api.DeviceBuffer.from_numpy(ctx, x) for x in flat + [ct]]
            if field == 1:
                for b, x in zip(bufs, flat + [ct]):
                    api._chk(api.lib().hg_field_encode(ctx.h, b.ptr, x.size // 4))
            return bufs[:-1], bufs[-1]
        resident = []
        for B in [int(b) for b in a.batches.split(",")]:
            # every proof has its own copy of the inputs: the verifier shares work only between proofs with the same tables
            while len(resident) < B:
                resident.append(upload())
            row = {"n": a.n, "field": "goldilocks" if field == 0 else "bn254", "batch": B, "host_proofs_per_s": 1.0 / host_s,
                   "host_cores_used": 1, "host_cpu_count": os.cpu_count()}
            for kind, ins_b, ct_b in (("resident", [r[0] for r in resident[:B]], [r[1] for r in resident[:B]]), ("host_vectors", [flat] * B, [ct] * B)):
                res = ver.verify_batch(ctx, ins_b, ct_b, [proof] * B)                      # warm-up, also sizes the pools
                assert all(ok for ok, _ in res), res[0]
                ts, reps = [], []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    ver.verify_batch(ctx, ins_b, ct_b, [proof] * B)
                    ts.append(time.perf_counter() - t0)
                    reps.append(ver._batch.timing())
                row[f"{kind}_proofs_per_s"] = B / min(ts)
                row[f"{kind}_ms_per_batch"] = 1e3 * min(ts)
                # host phases of hg_gkr_verify_batch (library timer): the replays alone, the device stages, closing the records
                best = reps[ts.index(min(ts))]
                row[f"{kind}_replay_ms_per_proof"] = best["replay_us"] / 1e3 / B
                row[f"{kind}_device_stages_ms_per_batch"] = best["device_us"] / 1e3
            # per-class device time and algorithmic bytes of one resident batch
            ctx.profile(True)
            ver.verify_batch(ctx, [r[0] for r in resident[:B]], [r[1] for r in resident[:B]], [proof] * B)
            prof = ctx.profile_read()
            row["device_ms_per_class"] = {k: round(v[1], 3) for k, v in prof.items() if v[0]}
            row["device_GB_per_class"] = {k: round(v[2] / 1e9, 3) for k, v in prof.items() if v[0]}
            ctx.profile(False)
            print(json.dumps(row), flush=True)
        ctx.close()


if __name__ == "__main__":
    main()
