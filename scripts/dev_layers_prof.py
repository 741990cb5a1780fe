"""Per-class kernel time of the full GKR proof (single stream, profiling mode)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
import hyper_greco_b200  # noqa
from hyper_greco_b200 import api
from hyper_greco_b200 import params
P = params.PARAMS[bench.DEFAULT_CONFIG]
ins, ct0is = bench.make_witness(bench.DEFAULT_CONFIG, 0)
ctx = api.Context(0)
prover = api.BfvSkEncryptProver(ctx, P)
flat = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
dev_inputs = [api.DeviceBuffer.from_numpy(ctx, np.array(v, dtype=np.uint64)) for v in flat]
d_ct = api.DeviceBuffer.from_numpy(ctx, np.array(ct0is, dtype=np.uint64))
prover.circuit.evaluate(dev_inputs)
tr0 = api.Keccak256Transcript()
point = tr0.squeeze_challenges(prover.ct0is_log2_size)
value = api.mle_eval_batch(ctx, d_ct, 1, prover.ct0is_log2_size, point)[0]
el = point.shape[1]
out_claims = [(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)]
def step():
    tr = api.Keccak256Transcript(); tr.squeeze_challenges(prover.ct0is_log2_size)
    prover.circuit.prove_gkr(out_claims, tr, api.MODE_PREFETCH)
    return tr.into_proof()
import hashlib
for _ in range(5): pr = step()
ctx.synchronize(); t0 = time.perf_counter()
for _ in range(20): step()
dt = (time.perf_counter() - t0) / 20
ctx.profile(True)
for _ in range(3): step()
prof = ctx.profile_read(); ctx.profile(False)
print(f"{dt*1e3:.3f} ms/proof sha={hashlib.sha256(pr).hexdigest()[:10]} " + " ".join(f"{k}={v[1]/3:.3f}" for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])[:12]))
