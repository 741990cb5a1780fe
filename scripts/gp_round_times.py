"""Device time of every grand-product and node-sumcheck launch of one full GKR proof, in launch order (torch.profiler, CUDA
activities; prefetch mode). Median over `--proofs` profiled proofs after warm-up.

    python scripts/gp_round_times.py [--proofs 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
import hyper_greco_b200  # noqa: E402,F401
from hyper_greco_b200 import api, params  # noqa: E402

PREFIXES = ("k_gp_fold_multi", "k_gp_tail", "k_prod_round_multi", "k_prod_tail", "k_copy_items")


def short(name):
    n = name.replace("hg::", "").replace("void ", "")
    return n.split("(")[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
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
        tr = api.Keccak256Transcript()
        tr.squeeze_challenges(prover.ct0is_log2_size)
        prover.circuit.prove_gkr(out_claims, tr, api.MODE_PREFETCH)
        ctx.synchronize()

    for _ in range(3):
        step()
    runs = []
    with tempfile.TemporaryDirectory() as td:
        for _ in range(a.proofs):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step()
            path = os.path.join(td, "t.json")
            prof.export_chrome_trace(path)
            ev = json.load(open(path))["traceEvents"]
            ks = sorted((e for e in ev if e.get("cat") == "kernel" and short(e["name"]).split("<")[0] in PREFIXES), key=lambda e: e["ts"])
            runs.append([(short(e["name"]), e["dur"]) for e in ks])
    n = min(len(r) for r in runs)
    lines = [f"# {torch.cuda.get_device_name(0)}; median of {a.proofs} proofs, us", ""]
    tot = {}
    for i in range(n):
        name = runs[0][i][0]
        us = statistics.median(r[i][1] for r in runs)
        tot[name.split("<")[0]] = tot.get(name.split("<")[0], 0.0) + us
        lines.append(f"{i:3d}  {us:9.1f}  {name}")
    lines.append("")
    for k, v in tot.items():
        lines.append(f"total {k}: {v:.1f} us")
    txt = "\n".join(lines)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
