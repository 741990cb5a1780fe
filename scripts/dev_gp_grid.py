"""Lasso-node proof time (device-resident input) and the hash / tree / grand-product class times."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
import hyper_greco_b200  # noqa
from hyper_greco_b200 import api
P, inp, bounds, segs, nv = bench.make_case(bench.DEFAULT_CONFIG, 0)
ctx = api.Context(0)
pp = api.LassoPreprocessing.preprocess(bounds)
node = api.LassoNode(ctx, pp, nv, segs)
buf = api.DeviceBuffer.from_numpy(ctx, inp)
ref = None
for _ in range(5):
    tr = api.Keccak256Transcript(); node.prove_claim_reduction(buf, tr, 0, n_inputs=inp.size)
proof = tr.into_proof()
import hashlib
t0 = time.perf_counter()
for _ in range(30):
    tr = api.Keccak256Transcript(); node.prove_claim_reduction(buf, tr, 0, n_inputs=inp.size)
dt = (time.perf_counter() - t0) / 30
ctx.profile(True)
for _ in range(3):
    tr = api.Keccak256Transcript(); node.prove_claim_reduction(buf, tr, 0, n_inputs=inp.size)
prof = ctx.profile_read(); ctx.profile(False)
gp = prof["sumcheck_grand_product"]
print(f"{dt*1e3:.3f} ms/proof, hash {prof['hash_build'][1]/3:.3f} tree {prof['product_tree'][1]/3:.3f} GP {gp[1]/3:.3f} ms, sha={hashlib.sha256(proof).hexdigest()[:12]}")
