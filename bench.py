#!/usr/bin/env python
"""Benchmark of the B200-native hyper-greco proving path (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py --gpus 1 --steps K --warmup W                 # our arm
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + the outputs of the last timed step, to compare two builds
    python bench.py --impl reference --gpus 1 --steps K --warmup W   # CPU arm: the oracle port on the host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU, weak scaling

    torchrun ... bench.py --gpus N --shard                         # extra: ONE Lasso-node proof split over N GPUs (strong scaling)

A step = one batch of `--inflight` independent proofs per GPU (default 4; each in its own context on its own host thread, so that
host work and PCIe copies of one proof overlap device work of the others); a proof = gkr::prove_gkr of the BFV SK-encryption
circuit (sk_encryption_circuit.rs:455-457) on a synthetic witness of the n=32768, k=16, Goldilocks parameter set (BASELINE.json
metric config). `value` = proofs/s over all GPUs; the latency of one proof alone is reported next to it. ONE JSON line on rank 0.
"""
import argparse
import gc
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.md rows "n=32768, 59, 16 - GKR prove": 5.06 s Goldilocks/Ext2, 28.8 s BN254 (reference README.md:44,56, Apple M1):
# the only published numbers for this metric; vs_baseline = value / these
PUBLISHED_PROOFS_PER_SEC = {"goldilocks": 1.0 / 5.06, "bn254": 1.0 / 28.8}
METRIC = "gkr_prove_proofs_per_sec"
UNIT = "proofs/s"
DEFAULT_CONFIG = "32768_16x59_65537"
NOMINAL_HBM_GBS = 8000.0   # the ~8 TB/s the north star quotes; the measured copy bandwidth is in MEASURED_PEAKS.json
WITNESS_POOL = 8           # distinct synthetic witnesses per rank (generated on the device, hg_bfv_witness_generate)
DUMP_LIMIT_BYTES = 64 << 20   # --dump-outputs writes at most this much


def bench_config(args, P, nv, m):
    """The `config` object of the JSON line: the SAME dict in both arms (our arm and --impl reference)."""
    fld = "goldilocks/ext2" if args.field == "goldilocks" else "bn254 Fr (E = F, 4x64 Montgomery)"
    return {
        "workload": f"gkr::prove_gkr of the BFV SK-encryption circuit n={P.N} k={P.K} {fld}: Lasso node (num_vars={nv}, memories={m}, C=4, M=65536) "
                    f"+ {2 * P.K + 1} FFT layers of 2^{P.log2_size} + {P.K} product layers + the Vanilla relay/scale/sum layers; a step = one batch of independent proofs per GPU",
        "scope": "the reference's `GKR prove` span (sk_encryption_circuit.rs:455-457): every node's claim reduction incl. LassoNode::polynomialize; "
                 "circuit values resident on the device (witness gen = circuit.evaluate is outside the span, as in the reference)",
        "params": args.config,
        "field": args.field,
        "parallelism": "independent proof instances: `proofs_in_flight_per_gpu` per GPU (one host thread + one context each), no data-path collective",
        "proofs_in_flight_per_gpu": max(1, args.inflight),
        "witness": f"{WITNESS_POOL} synthetic witnesses per rank (seeds {WITNESS_POOL}*rank ..), generated on the device (hg_bfv_witness_generate) and kept in pinned "
                   "host memory: slot k proves witness k in the resident region, every slot cycles through all of them in the end-to-end region",
        "cache": "working set ~4 GB per proof >> 126 MB L2, no explicit flush between steps",
        "harness": "python gc paused inside the timed regions (the caller in production is Rust)",
    }


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (NVML every 100 ms; faster polling measurably slows the
    launch path through the driver lock)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz, self._stop, self._t = index, [], set(), None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80,
                 "sync_boost": 0x10, "applications_clocks_setting": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


FIELD_ID = {"goldilocks": 0, "bn254": 1}


def make_witness(name, seed, field="goldilocks"):
    """(python-int inputs dict, ct0is) of one synthetic witness (hyper-greco_b200/witness.py, distribution of scripts/circuit_sk.py:29-140)."""
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import params, witness
    P = params.PARAMS[name]
    a = witness.synth_witness(P, seed, p=witness.BN_R) if field == "bn254" else witness.synth_witness(P, seed)
    return witness.get_inputs(P, a)


def to_limbs(v, field):
    """python ints -> contiguous uint64 limbs ([n] Goldilocks, [4n] BN254: canonical little-endian)"""
    import numpy as np
    if field == "goldilocks":
        return np.array(v, dtype=np.uint64)
    return np.array([[(int(x) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for x in v], dtype=np.uint64).reshape(-1)


def host_vectors(ins, ct0is, field):
    flat = [ins["s"], ins["e"], ins["k1"]] + list(ins["ais"]) + list(ins["r1is"]) + [ins["r2is"]]
    return [to_limbs(v, field) for v in flat], to_limbs(ct0is, field)


def make_case(name, seed):
    """Lasso-node input of one synthetic witness (used by scripts/ and the node-level tools)."""
    import numpy as np
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import params, witness
    P = params.PARAMS[name]
    args = witness.synth_witness(P, seed)
    inp = np.array(witness.lasso_inputs(P, args), dtype=np.uint64)
    return P, inp, witness.lasso_lookup_bounds(P), witness.lasso_lookup_segments(P), witness.lasso_num_vars(P)


def oracle_case(hgo, bounds, segs):
    import numpy as np
    opp = hgo.Preprocessing(bounds)
    rows = np.concatenate([np.full(l, opp.lookup_index(b), np.int32) for b, l in segs])
    return opp, rows


def run_reference(args):
    """CPU arm: the reference's own implementation cannot be built here (Rust nightly + un-vendored git deps, SURVEY F1/F2),
    so this times the oracle port (oracle/protocol.hpp + oracle/gkr.hpp, OpenMP over all host cores) on the same workload:
    the `GKR prove` span with the circuit already evaluated. W warm-up proofs, then K timed ones; if that does not fit in
    ~4.5 minutes K (then W) is reduced and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import params, witness
    from oracle import hgo
    hgo.build()
    P = params.PARAMS[args.config]
    fid = FIELD_ID[args.field]
    ins, ct0is = make_witness(args.config, 0, args.field)
    opp = hgo.Preprocessing(witness.lasso_lookup_bounds(P))
    nv = witness.lasso_num_vars(P)
    hgo.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host core
    cores = hgo.num_threads()
    if fid == 0:
        prep = hgo.bfv_prepare(fid, P, ins, ct0is)
        one = lambda: hgo.bfv_prove_prepared(prep)
    else:   # the prepared-session API of the oracle is Goldilocks only: BfvEncrypt::prove as a whole (circuit.evaluate included, ~3 % of it)
        one = lambda: hgo.bfv_prove(fid, P, ins, ct0is, cap=1 << 26)
    t0 = time.perf_counter()
    one()
    t1 = time.perf_counter() - t0
    budget = 270.0
    want_w = max(args.warmup, 1)
    steps, warm = args.steps, want_w
    if (warm - 1 + steps) * t1 > budget:
        warm = 1
        steps = max(1, min(args.steps, int(budget / max(t1, 1e-3)) - 1))
    for _ in range(warm - 1):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    v = steps / dt
    capped = steps < args.steps or warm < want_w
    sample = f"{steps} full proofs of the same workload after {warm} warm-up proof(s) (first one {t1:.1f}s)" + \
             (f"; --steps {args.steps} --warmup {args.warmup} reduced to fit ~4.5 min" if capped else "")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1000.0 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": v / PUBLISHED_PROOFS_PER_SEC[args.field] if args.config == DEFAULT_CONFIG else None, "dtype": "u64" if fid == 0 else "u256", "data": "synthetic",
            "config": bench_config(args, P, nv, opp.num_memories),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


class HostWitness:
    """One witness as the caller holds it: the get_inputs vectors (sk_encryption_circuit.rs:365-415) and ct0is in ONE pinned block."""

    def __init__(self, np, torch, host_np, ct_np):
        n_in = sum(v.size for v in host_np)
        self.pinned = torch.empty(n_in + ct_np.size, dtype=torch.int64).pin_memory()
        h_all = self.pinned.numpy().view(np.uint64)
        self.views, off = [], 0
        for v in host_np:
            h_all[off:off + v.size] = v
            self.views.append(h_all[off:off + v.size])
            off += v.size
        self.ct = h_all[n_in:]
        self.ct[:] = ct_np
        self.bytes = int(h_all.nbytes)


class ProofSlot:
    """One proof in flight: its own hg_ctx (streams) and prover (6 GB of device buffers for Goldilocks); witness k resident."""

    def __init__(self, api, np, P, pool, k, device, field_id):
        self.api, self.np, self.pool, self.k = api, np, pool, k
        self.ctx = api.Context(device, field_id)
        self.prover = api.BfvSkEncryptProver(self.ctx, P)             # setup + configure (sk_encryption_circuit.rs:319-363)
        w = pool[k % len(pool)]
        self.dev_inputs = [api.DeviceBuffer.from_field(self.ctx, v) for v in w.views]
        self.d_ct = api.DeviceBuffer.from_field(self.ctx, w.ct)
        self.prover.circuit.evaluate(self.dev_inputs)                 # witness gen (outside the `GKR prove` span, :439-453)
        self.out_claims = self.output_claims(api.Keccak256Transcript(field_id))
        self.field_id = field_id
        self.e2e_i = k

    def output_claims(self, tr):
        L = self.prover.ct0is_log2_size
        point = tr.squeeze_challenges(L)                              # :445
        value = self.api.mle_eval_batch(self.ctx, self.d_ct, 1, L, point)[0]   # :446
        el = point.shape[1]
        return [(self.np.zeros((0, el), self.np.uint64), self.np.zeros(el, self.np.uint64)), (point, value)]

    def resident(self):
        """the `GKR prove` span: gkr::prove_gkr on device-resident circuit values. What its caller receives (the transcript holding
        the proof, the input claims) is kept in `last` until the next proof of this slot."""
        tr = self.api.Keccak256Transcript(self.field_id)
        tr.squeeze_challenges(self.prover.ct0is_log2_size)
        self.last = (tr, self.prover.circuit.prove_gkr(self.out_claims, tr, self.api.MODE_PREFETCH))
        return tr

    def e2e(self, which=None):
        """BfvEncrypt::prove from HOST vectors (pinned): H2D of the witness vectors and of ct0is, circuit.evaluate, output claim,
        prove_gkr, proof bytes on the host. Every call takes the next witness of the pool."""
        if which is None:
            self.e2e_i = (self.e2e_i + 1) % len(self.pool)
            which = self.e2e_i
        w = self.pool[which]
        return self.prover.prove_host(w.views, w.ct)[0]

    def restore_resident(self):
        """prove_host re-evaluated the circuit on another witness: put this slot's own witness back"""
        self.prover.circuit.evaluate(self.dev_inputs)
        self.ctx.synchronize()

    def close(self):
        self.prover.circuit.free()
        self.prover.lasso.free()
        self.ctx.close()


def run_slots(slots, fn_name, n):
    """every slot runs n proofs on its own host thread (the C calls release the GIL); returns when all are done"""
    if len(slots) == 1:
        f = getattr(slots[0], fn_name)
        for _ in range(n):
            f()
        return
    errs = []

    def work(s):
        try:
            f = getattr(s, fn_name)
            for _ in range(n):
                f()
        except Exception as e:  # pragma: no cover
            errs.append(e)

    ths = [threading.Thread(target=work, args=(s,)) for s in slots]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:
        raise errs[0]


def measure_sharded(api, np, torch, dist, slot, host_w, steps, warmup, rank, world, barrier):
    """BASELINE.json config 4: ONE gkr::prove_gkr split over all ranks (hg_gkr_prove_shard_dev: generic node sumchecks by node, the
    Lasso node by grand-product vectors / openings / counter slots; exchange = NCCL all-gather of the message buffers + one
    merge kernel, rank 0 serialises). Every rank holds the same witness. Wall clock of K proofs between barriers, max over ranks;
    the same proof on rank 0 alone right after, for the speed-up."""
    prover, ctx = slot.prover, slot.ctx
    prover.circuit.evaluate_host(host_w.views)                       # the SAME witness on every rank
    d_ct = api.DeviceBuffer.from_field(ctx, host_w.ct)
    L = prover.ct0is_log2_size
    tr0 = api.Keccak256Transcript(slot.field_id)
    point = tr0.squeeze_challenges(L)
    value = api.mle_eval_batch(ctx, d_ct, 1, L, point)[0]
    el = point.shape[1]
    claims = [(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)]
    ex = api.ShardExchange(ctx, prover.circuit.shard_words)
    last = {}
    split_emit = os.environ.get("HG_SHARD_SPLIT_EMIT", "1") != "0" and world > 1

    def step():
        tr = api.Keccak256Transcript(slot.field_id)
        tr.squeeze_challenges(L)
        if split_emit:   # every rank serialises one range of the proof, rank 0 appends the gathered ranges
            ex.run(lambda r, w, ptr, cap: prover.circuit.prove_gkr_shard_dev(claims, tr, r, w, ptr, cap), None,
                   emit_part=prover.circuit.emit_shard_part_dev, transcript=tr)
        else:
            ex.run(lambda r, w, ptr, cap: prover.circuit.prove_gkr_shard_dev(claims, tr, r, w, ptr, cap), prover.circuit.emit_shard_dev)
        last["tr"] = tr

    for _ in range(max(warmup, 3) + 10):
        step()
    gc.collect()
    gc.disable()   # a generation-2 collection of the harness's Python heap inside the loop cost 25 ms once per measurement (profiles/r2_experiments.md)
    barrier()
    w0 = time.perf_counter()
    for _ in range(steps):
        step()
    barrier()
    gc.enable()
    t = torch.tensor([time.perf_counter() - w0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_sharded = 1000.0 * float(t[0]) / steps
    res = None
    phases = getattr(ex, "phases", None)
    if phases is not None:
        print(f"[shard rank {rank}] phases of the last proof: " + json.dumps({k: round(v, 3) for k, v in phases.items()}), file=sys.stderr)
    if rank == 0:
        proof = last["tr"].into_proof()

        def single():
            tr = api.Keccak256Transcript(slot.field_id)
            tr.squeeze_challenges(L)
            prover.circuit.prove_gkr(claims, tr, api.MODE_PREFETCH)
            return tr
        for _ in range(5):
            tr1 = single()
        w0 = time.perf_counter()
        for _ in range(steps):
            single()
        ms_one = 1000.0 * (time.perf_counter() - w0) / steps
        res = {"gpus": world, "ms_per_proof": ms_sharded, "one_gpu_ms_per_proof": ms_one, "speedup_vs_1gpu": ms_one / ms_sharded,
               "bytes_equal": tr1.into_proof() == proof, "steps": steps,
               "partition": "generic node sumchecks by node (q % gpus), Lasso node by grand-product vectors, openings and counter slots; polynomialize replicated",
               "collective": f"one NCCL all_gather of {8 * prover.circuit.shard_words} bytes per rank per proof (message buffers only) + one merge kernel; "
                             + ("every rank serialises one range of the proof (hg_gkr_emit_shard_part_dev), one all_gather of the byte ranges, rank 0 appends them"
                                if split_emit else "rank 0 serialises (one D2H of the same size)"),
               "timing": "wall clock between barriers, max over ranks (the step ends with host-side serialisation on rank 0)"}
    barrier()
    d_ct.free()
    return res


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, params, witness

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api.lib()
    fid = FIELD_ID[args.field]
    P = params.PARAMS[args.config]
    nv = witness.lasso_num_vars(P)

    B = max(1, args.inflight)
    pool_n = max(1, min(WITNESS_POOL, args.pool))
    # the witness pool: generated on the device (scripts/circuit_sk.py:72-140 as kernels), downloaded once into pinned host memory
    # (the end-to-end region starts from HOST vectors, as BfvEncrypt::prove does). Same seeds -> same witnesses as make_witness.
    pool = []
    gen_ctx = api.Context(local, fid)
    t_gen = time.perf_counter()
    gen_dev_s = 0.0
    for k in range(pool_n):
        t_g = time.perf_counter()
        dev, d_ct = witness.synth_witness_device(gen_ctx, P, WITNESS_POOL * rank + k)
        gen_dev_s += time.perf_counter() - t_g
        lens = [2 * P.N] * (3 + 2 * P.K) + [P.K * P.N]
        host = [b.to_field(n).reshape(-1) for b, n in zip(dev, lens)]
        pool.append(HostWitness(np, torch, host, d_ct.to_field(P.K * 2 * P.N).reshape(-1)))
        for b in dev[:3] + [dev[3].base, dev[3 + P.K].base, dev[-1], d_ct]:
            b.free()
    witness_gen_ms = {"generate_on_device_ms": 1000.0 * gen_dev_s / pool_n, "with_download_to_pinned_host_ms": 1000.0 * (time.perf_counter() - t_gen) / pool_n,
                      "note": "per witness; numpy draws + hg_bfv_witness_generate (synchronous), then the copy into the host pool of the end-to-end region"}
    gen_ctx.close()
    n_in_bytes = pool[0].bytes
    slots = [ProofSlot(api, np, P, pool, k, local, fid) for k in range(B)]
    s0 = slots[0]
    ctx, prover, pp = s0.ctx, s0.prover, s0.prover.pp

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_resident = s0.resident

    # device spin-up (setup, untimed): the first ~20 proofs after process start run up to 12 % slower (first-touch of the work
    # buffers, lazily created kernels/attributes, challenge-chain cache); a prover service is measured in steady state
    spin_up = 0
    t_spin = time.perf_counter()
    while spin_up < 10 or time.perf_counter() - t_spin < 0.4:
        run_slots(slots, "resident", 1)
        spin_up += 1
    warm = max(args.warmup, 3)
    run_slots(slots, "resident", warm)
    tr = step_resident()
    proof_len = len(tr.into_proof())
    host_phases = prover.circuit.timing()
    l0 = ctx.launch_count
    step_resident()
    launches_per_proof = ctx.launch_count - l0

    # ---- single-proof latency (one proof at a time on this GPU), CUDA events on the library's stream
    ext = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    n_lat = max(30, args.steps)
    for _ in range(n_lat):
        step_resident()
    e1.record(ext)
    barrier()
    latency_ms = e0.elapsed_time(e1) / n_lat

    # ---- the same proof in INTERACTIVE mode (one device->host->device round trip per squeeze: what a caller-owned transcript that
    # absorbs its messages gets, INTEGRATION.md section 3); single GPU only, a few proofs, outside every timed region
    interactive_ms = None
    if world == 1:
        def interactive():
            tr_i = api.Keccak256Transcript(fid)
            tr_i.squeeze_challenges(prover.ct0is_log2_size)
            prover.circuit.prove_gkr(s0.out_claims, tr_i, api.MODE_INTERACTIVE)
            return tr_i
        same_bytes = interactive().into_proof() == tr.into_proof()
        w0 = time.perf_counter()
        for _ in range(3):
            interactive()
        interactive_ms = {"single_proof_latency_ms": 1000.0 * (time.perf_counter() - w0) / 3, "bytes_equal_prefetch": same_bytes,
                          "note": "HG_MODE_INTERACTIVE: one round trip per challenge (1 534 per proof), sequential per-layer launches"}

    # ---- timed region: exactly K steps; a step = one batch of B independent proofs, one per in-flight slot (slot k proves witness
    # k). Every slot ends each proof with a stream synchronise, so the device is idle at both events; events on torch's current
    # stream between two device-wide synchronisations measure the device time of the whole region. Max over ranks.
    sampler = ClockSampler(local)
    gc.collect()
    gc.disable()   # re-enabled after the end-to-end region: the harness's garbage collector is not part of the product
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    w0 = time.perf_counter()
    run_slots(slots, "resident", args.steps)
    torch.cuda.synchronize()
    e1.record()
    barrier()
    wall = time.perf_counter() - w0
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    last_step = [s.last for s in slots]
    t = torch.tensor([ms, wall * 1000.0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, wall_ms = float(t[0]), float(t[1])
    value = world * B * args.steps / (ms_total / 1000.0)

    # ---- end to end through the C ABI with HOST buffers (H2D of the inputs and D2H of the proof messages inside); every slot
    # walks through the witness pool, so consecutive proofs of a slot are of different witnesses
    run_slots(slots, "e2e", 3)
    barrier()
    w0 = time.perf_counter()
    run_slots(slots, "e2e", args.steps)
    barrier()
    e2e_wall = time.perf_counter() - w0
    t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t[0])
    w0 = time.perf_counter()
    for _ in range(n_lat):
        s0.e2e()
    e2e_latency_ms = 1000.0 * (time.perf_counter() - w0) / n_lat
    gc.enable()
    s0.restore_resident()

    line = None
    roofline = cpu = None
    if rank == 0:
        # ---- roofline of the dominant kernel class: CUDA events around every launch, separate pass right after the timed one
        # (the start event of a launch executes as soon as it is recorded on the idle profiling stream, so a host hiccup between the
        # record and the launch lands in that launch's time: every proof is profiled on its own and the per-class MEDIAN of the
        # proofs is reported, scaled back to prof_steps so the arithmetic below is unchanged)
        prof_steps = 5
        runs = []
        for _ in range(prof_steps):
            ctx.profile(True)
            step_resident()
            runs.append(ctx.profile_read())
            ctx.profile(False)
        prof = {k: (sum(r[k][0] for r in runs), statistics.median(r[k][1] for r in runs) * prof_steps, sum(r[k][2] for r in runs)) for k in runs[0]}
        dom = max(prof.items(), key=lambda kv: kv[1][1])
        dn, (dl, dms, dby) = dom
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md 6.65 TB/s)"
        achieved = (dby / 1e9) / (dms / 1e3) if dms > 0 else 0.0
        traffic = traffic_step = None
        try:   # ncu DRAM bytes of the same kernels (profiles/traffic.json, written by scripts/make_profiles.py from an ncu run of this command)
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dn)
            traffic, traffic_step = tj["bytes_per_launch"], tj["bytes_per_step"]
        except Exception:
            pass
        total_ms = sum(v[1] for v in prof.values())
        total_gb = sum(v[2] for v in prof.values()) / prof_steps / 1e9
        per_class = {k: {"launches": v[0] / prof_steps, "ms": v[1] / prof_steps, "alg_GB": v[2] / prof_steps / 1e9,
                         "GBps": (v[2] / 1e9) / (v[1] / 1e3) if v[1] > 0 else None} for k, v in prof.items()}
        # the grand-product pipeline as a whole (SURVEY 8d rows "GP tree", "hash build", "GP sumchecks"): since round 0 of every layer
        # sumcheck is sampled by the hash / tree builders (gp_fused.cuh), the three classes share that work
        gp_names = ("hash_build", "product_tree", "sumcheck_grand_product")
        gp_ms = sum(per_class[k]["ms"] for k in gp_names if k in per_class)
        gp_gb = sum(per_class[k]["alg_GB"] for k in gp_names if k in per_class)
        roofline = {"bound": "hbm", "kernel": dn, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                    "frac_vs_nominal_8TBs": achieved / NOMINAL_HBM_GBS, "peak_nominal": NOMINAL_HBM_GBS,
                    "traffic": traffic, "traffic_bytes_per_proof": traffic_step, "algorithmic_bytes_per_launch": dby / max(dl, 1),
                    "algorithmic_bytes_per_proof": dby / prof_steps, "peak_source": peak_src,
                    "launches_per_proof": dl / prof_steps, "avg_launch_us": 1000.0 * dms / max(dl, 1),
                    "share_of_proof_kernel_time": dms / total_ms if total_ms else None,
                    "timing": f"CUDA events around every launch on the launching stream, {prof_steps} proofs profiled one by one right after the timed region, "
                              "per-class median over the proofs",
                    "note": "rounds >= 1 of the layer sumchecks; round 0 (1.73 GB of SURVEY 8d's 10.38 GB for this class) is sampled by the hash / tree builders and "
                            "needs no pass of its own, see grand_product_pipeline",
                    "grand_product_pipeline": {"classes": list(gp_names), "ms": gp_ms, "alg_GB": gp_gb, "GBps": gp_gb / (gp_ms / 1e3) if gp_ms else None,
                                               "frac": (gp_gb / (gp_ms / 1e3)) / peak if gp_ms and peak else None,
                                               "survey_8d_alg_GB": gp_gb + 1.7304, "frac_with_survey_8d_bytes": ((gp_gb + 1.7304) / (gp_ms / 1e3)) / peak if gp_ms and peak and args.config == DEFAULT_CONFIG and fid == 0 else None},
                    "per_class": per_class,
                    "whole_proof_alg_GB": total_gb,
                    "whole_proof_kernel_ms_single_stream": total_ms / prof_steps,
                    "whole_proof_frac_single_stream": total_gb / (total_ms / prof_steps / 1e3) / peak if total_ms else None,
                    "whole_proof_frac_inflight": total_gb / ((ms_total / (args.steps * B)) / 1e3) / peak,
                    "whole_proof_frac_note": "single_stream: bytes / summed kernel time of ONE proof run alone (profiling pass); inflight: the same bytes / time per proof of the "
                                             "timed region, where kernels of several proofs overlap"}
        # ---- CPU baseline: the oracle port on this box's host cores, one full proof (N=1 only)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import hgo
            hgo.build()
            hgo.set_num_threads(os.cpu_count() or 1)
            ins0, ct0 = make_witness(args.config, WITNESS_POOL * rank, args.field)   # numpy restatement of the same witness (seed 0)
            if fid == 0:
                sess = hgo.bfv_prepare(fid, P, ins0, ct0)
                t0 = time.perf_counter()
                oproof = sess.prove()
            else:   # BN254: the oracle's one-shot BfvEncrypt::prove (circuit.evaluate included)
                t0 = time.perf_counter()
                oproof = hgo.bfv_prove(fid, P, ins0, ct0, cap=1 << 26)
            dt = time.perf_counter() - t0
            same = oproof == s0.e2e(0)
            cpu = {"value": 1.0 / dt, "unit": UNIT, "cores": hgo.num_threads(), "kind": "port",
                   "sample": f"1 full proof of witness 0 ({dt:.1f}s); GPU proof bytes == CPU proof bytes: {same}"}
    # ---- one proof over all GPUs (BASELINE.json config 4), reported inside the same line
    shard = None
    if world > 1 and not args.no_shard:
        shared_w = HostWitness(np, torch, *host_vectors(*make_witness(args.config, 10_000, args.field), args.field))   # the same witness on every rank
        shard = measure_sharded(api, np, torch, dist, s0, shared_w, max(10, args.steps), warm, rank, world, barrier)
    if rank == 0:
        node_ch = node_chal_bytes(nv) * (1 if fid == 0 else 1)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": ms_total / args.steps, "ms_per_proof": ms_total / (args.steps * B), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": value / PUBLISHED_PROOFS_PER_SEC[args.field] if args.config == DEFAULT_CONFIG else None,
                "vs_baseline_note": "published: 5.06 s (Goldilocks) / 28.8 s (BN254) per proof on an Apple M1 (reference README.md:44,56, BASELINE.md); other hardware",
                "dtype": "u64" if fid == 0 else "u256", "data": "synthetic", "config": bench_config(args, P, nv, pp.num_memories), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(B * (n_in_bytes + node_ch + 4096)),
                        "d2h_bytes_per_step": int(B * proof_len * 2), "single_proof_latency_ms": e2e_latency_ms},
                "gpu_launches": int(launches_per_proof * args.steps * B), "gpu_launches_per_proof": int(launches_per_proof),
                "single_proof_latency_ms": latency_ms, "interactive_mode": interactive_ms, "wall_ms_per_step": wall_ms / args.steps, "proof_bytes": proof_len, "spin_up_steps": spin_up, "witness_gen_ms_per_witness": witness_gen_ms,
                "host_phases_us": host_phases, "roofline": roofline, "cpu_baseline": cpu, "shard": shard}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step, f"rank{rank}_" if world > 1 else "")
    barrier()
    for s in slots:
        s.close()
    if world > 1:
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))


def u64_as_f64(words):
    """uint64 limbs -> float64 [n, 2] (low, high 32 bits of each limb): exact, so two dumps can be compared value for value"""
    import numpy as np
    w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1)
    return np.stack([w & np.uint64(0xFFFFFFFF), w >> np.uint64(32)], -1).astype(np.float64)


def dump_outputs(out_dir, last_step, prefix=""):
    """--dump-outputs: what every in-flight proof of the last timed step handed to its caller, as <prefix>proof_<slot>.npy (the proof
    bytes, float32) and <prefix>input_claims_<slot>.npy (point then value of every claim on every input node, in node order, through
    u64_as_f64). Slots are written in order while the total stays within DUMP_LIMIT_BYTES."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for k, (tr, claims) in enumerate(last_step):
        proof = np.frombuffer(tr.into_proof(), np.uint8).astype(np.float32)
        words = [a.reshape(-1) for node in claims for pt, val in node for a in (pt, val)]
        cl = u64_as_f64(np.concatenate(words) if words else np.zeros(0, np.uint64))
        if total + proof.nbytes + cl.nbytes > DUMP_LIMIT_BYTES:
            print(f"bench.py: --dump-outputs stops after {k} of {len(last_step)} slots ({DUMP_LIMIT_BYTES >> 20} MB)", file=sys.stderr)
            break
        np.save(os.path.join(out_dir, f"{prefix}proof_{k}.npy"), proof)
        np.save(os.path.join(out_dir, f"{prefix}input_claims_{k}.npy"), cl)
        total += proof.nbytes + cl.nbytes


def run_shard(args):
    """`--shard`: only the sharded measurement of run_ours (ONE gkr::prove_gkr over the N ranks)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import hyper_greco_b200  # noqa: F401
    from hyper_greco_b200 import api, params, witness

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fid = FIELD_ID[args.field]
    P = params.PARAMS[args.config]
    w = HostWitness(np, torch, *host_vectors(*make_witness(args.config, 10_000, args.field), args.field))
    slot = ProofSlot(api, np, P, [w], 0, local, fid)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    res = measure_sharded(api, np, torch, dist, slot, w, args.steps, max(args.warmup, 3), rank, world, barrier)
    if rank == 0:
        print(json.dumps({"metric": "gkr_prove_sharded_ms_per_proof", "value": res["ms_per_proof"], "unit": "ms", "n_gpus": world, "steps": args.steps,
                          "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_proof"], "higher_is_better": False, "scaling": "strong",
                          "dtype": "u64" if fid == 0 else "u256", "data": "synthetic",
                          "config": bench_config(args, P, witness.lasso_num_vars(P), slot.prover.pp.num_memories), "shard": res}))
    barrier()
    slot.close()
    dist.destroy_process_group()


def node_chal_bytes(nv, lm=16):
    gp = lambda k: sum(1 + ((1 + j) if j else 0) for j in range(k))
    return 16 * (2 * nv + 2 + gp(nv) + gp(lm))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=DEFAULT_CONFIG)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inflight", type=int, default=4, help="independent proofs in flight per GPU (a step = one batch of that many proofs)")
    ap.add_argument("--shard", action="store_true", help="only the sharded measurement: ONE gkr::prove_gkr split over the N GPUs (strong scaling)")
    ap.add_argument("--no-shard", action="store_true", help="skip the sharded measurement that a multi-GPU run adds to its line")
    ap.add_argument("--field", default="goldilocks", choices=["goldilocks", "bn254"], help="BASELINE.json config 5: --field bn254")
    ap.add_argument("--pool", type=int, default=WITNESS_POOL, help="distinct witnesses per rank (<= %d)" % WITNESS_POOL)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what every proof of the last timed step returned "
                    "as DIR/proof_<slot>.npy and DIR/input_claims_<slot>.npy (the inputs are the same from run to run with the same arguments)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.shard):
        ap.error("--dump-outputs writes the outputs of the default GPU run, not of --impl reference or --shard")
    if args.impl == "reference":
        run_reference(args)
    elif args.shard:
        run_shard(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
