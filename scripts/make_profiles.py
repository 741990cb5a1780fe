"""Turns the ncu captures brought back in gpurun_out/ into the tracked summaries under profiles/ (TAG = r2 unless given as argv[1]).

    gpurun_out/TAG_launches.csv : ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none
                                  -c 900 --csv python bench.py --steps 1 --warmup 3 --no-cpu-baseline --inflight 1 --pool 1
    gpurun_out/TAG_*.ncu-rep    : ncu --set full --clock-control none --import-source on -k regex:... python scripts/dev_gp_grid.py
(the exact commands are scripts/gpu_profile.sh). Writes profiles/TAG_launch_list.md, profiles/traffic.json, profiles/TAG_ncu_gp_kernels.txt."""
import collections
import csv
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLASSES = [
    ("sumcheck_grand_product", r"k_gp_fold_multi|k_gp_tail"),
    ("misc", r"k_gp_coeffs_multi"),
    ("sumcheck_collation", r"k_coll_round|k_prod_tail_one|k_sc_round|k_fold_final|k_prod_mid_one"),
    ("gkr_layer_sumcheck", r"k_prod_round_multi|k_prod_tail|k_copy_items|k_fold_items"),
    ("gkr_layer_weights", r"k_eq_split_multi|k_eq_accumulate|k_wiring_gather|k_wiring_runs|k_concat_items|k_ext_split|k_ext_merge|k_dot_wconst"),
    ("counters", r"k_cnt_"),
    ("hash_build", r"k_hash_"),
    ("product_tree", r"k_tree_"),
    ("mle_dot", r"k_dot_eq"),
    ("eq_build", r"k_eq_split<"),
    ("ntt", r"k_ntt_"),
    ("polynomialize", r"k_polynomialize"),
]


def classify(name):
    for cls, pat in CLASSES:
        if re.search(pat, name):
            return cls
    return "other"


def main():
    TAG = sys.argv[1] if len(sys.argv) > 1 else "r2"
    src = os.path.join(ROOT, "gpurun_out", f"{TAG}_launches.csv")
    lines = [l for l in open(src) if not l.startswith("==")]
    byid = collections.OrderedDict()
    for x in csv.DictReader(lines):
        d = byid.setdefault(int(x["ID"]), {"name": x["Kernel Name"], "grid": x["Grid Size"], "block": x["Block Size"]})
        d[x["Metric Name"]] = float(x["Metric Value"].replace(",", ""))
    ids = list(byid)
    starts = [i for i in ids if "k_polynomialize" in byid[i]["name"]]
    a, b = starts[3], starts[4]   # the 4th proof of the run: after the 3 warm-up proofs, device-resident values, no evaluate in between
    step = [byid[i] for i in range(a, b)]
    total = sum(k["gpu__time_duration.sum"] for k in step)
    per_cls = collections.OrderedDict()
    per_kernel = collections.OrderedDict()
    for k in step:
        nm = re.sub(r"^void ", "", k["name"])
        nm = re.sub(r"\(.*", "", nm)
        for key, agg in ((classify(nm), per_cls), (nm, per_kernel)):
            e = agg.setdefault(key, [0, 0.0, 0.0, 0.0])
            e[0] += 1
            e[1] += k["gpu__time_duration.sum"]
            e[2] += k["dram__bytes_read.sum"]
            e[3] += k["dram__bytes_write.sum"]
    bench = None
    try:
        bench = json.loads(open(os.path.join(ROOT, "profiles", f"{TAG}_bench_ours.json")).read().strip().splitlines()[-1])
    except Exception:
        pass
    out = [f"# Launch list of one proof ({TAG}, final state)", "",
           "Command (on a B200 through gpurun): `ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum "
           f"--clock-control none -c 900 --csv --log-file gpurun_out/{TAG}_launches.csv python bench.py --steps 1 --warmup 3 --no-cpu-baseline --inflight 1 --pool 1`.",
           f"Rows below: launches {a}..{b - 1} of that run = the 4th `gkr::prove_gkr` (n=32768, k=16, Goldilocks), {len(step)} launches, "
           f"{total / 1e6:.3f} ms summed kernel time. Under ncu every launch is serialised and runs cold, so only the SHARES are comparable "
           f"with the CUDA-event numbers of `bench.py` (last column, `roofline.per_class` of profiles/{TAG}_bench_ours.json, where the same "
           "kernels run back to back on one stream in profiling mode).", "",
           "| class | launches | ncu time (us) | share | DRAM read (MB) | DRAM write (MB) | bench.py events: ms, share |", "|---|---|---|---|---|---|---|"]
    btot = sum(v["ms"] for v in bench["roofline"]["per_class"].values()) if bench else None
    for cls, e in sorted(per_cls.items(), key=lambda kv: -kv[1][1]):
        bcol = ""
        if bench and cls in bench["roofline"]["per_class"]:
            bm = bench["roofline"]["per_class"][cls]["ms"]
            bcol = f"{bm:.3f}, {100 * bm / btot:.1f} %"
        out.append(f"| {cls} | {e[0]} | {e[1] / 1e3:.1f} | {100 * e[1] / total:.1f} % | {e[2] / 1e6:.1f} | {e[3] / 1e6:.1f} | {bcol} |")
    out += ["", "| kernel | launches | ncu time (us) | DRAM read (MB) | DRAM write (MB) |", "|---|---|---|---|---|"]
    for nm, e in sorted(per_kernel.items(), key=lambda kv: -kv[1][1]):
        out.append(f"| `{nm}` | {e[0]} | {e[1] / 1e3:.1f} | {e[2] / 1e6:.1f} | {e[3] / 1e6:.1f} |")
    out += ["", "Every launch in order:", "", "| # | kernel | grid | block | us | read MB | write MB |", "|---|---|---|---|---|---|---|"]
    for n, k in enumerate(step):
        nm = re.sub(r"\(.*", "", re.sub(r"^void ", "", k["name"]))
        out.append(f"| {n} | `{nm}` | {k['grid']} | {k['block']} | {k['gpu__time_duration.sum'] / 1e3:.1f} | {k['dram__bytes_read.sum'] / 1e6:.2f} | {k['dram__bytes_write.sum'] / 1e6:.2f} |")
    open(os.path.join(ROOT, "profiles", f"{TAG}_launch_list.md"), "w").write("\n".join(out) + "\n")
    traffic = {"_comment": "DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum, ncu) of one proof per kernel class; bench.py reports "
                           "roofline.traffic = bytes per launch of the dominant class (class total / launches), like roofline.achieved is per launch",
               "_source": f"gpurun_out/{TAG}_launches.csv via scripts/make_profiles.py"}
    for cls, e in per_cls.items():
        traffic[cls] = {"launches": e[0], "bytes_per_step": e[2] + e[3], "bytes_per_launch": (e[2] + e[3]) / e[0]}
    json.dump(traffic, open(os.path.join(ROOT, "profiles", "traffic.json"), "w"), indent=1)
    keep = re.compile(r"k_gp_|k_hash_|k_tree_|gpu__time_duration.sum|dram__bytes_(read|write).sum |gpu__dram_throughput.avg.pct|sm__throughput.avg.pct|launch__registers_per_thread |"
                      r"launch__grid_size|launch__occupancy_limit_registers|sm__warps_active.avg.pct|smsp__inst_executed.sum |sm__pipe_(alu|fma)_cycles_active.avg.pct_of_peak_sustained_active|"
                      r"smsp__issue_active.avg.pct|smsp__average_warps_issue_stalled_(barrier|dispatch_stall|long_scoreboard|math_pipe_throttle|not_selected|wait|short_scoreboard|no_instruction)_per_issue_active|"
                      r"sm__inst_executed_pipe_(alu|fma|fmaheavy|lsu).sum |local_(load|store)")
    txt = []
    for rep_name in sorted(os.listdir(os.path.join(ROOT, "gpurun_out"))):
        if rep_name.startswith(TAG + "_") and rep_name.endswith(".ncu-rep"):
            raw = subprocess.run(["ncu", "-i", os.path.join(ROOT, "gpurun_out", rep_name), "--page", "raw"], capture_output=True, text=True).stdout
        elif rep_name.startswith(TAG + "_") and rep_name.endswith("_raw.txt"):   # `ncu -i ... --page raw` already run on the box
            raw = open(os.path.join(ROOT, "gpurun_out", rep_name)).read()
        else:
            continue
        txt += [f"===== {rep_name}: ncu --set full --clock-control none --import-source on (scripts/gpu_profile.sh), python scripts/dev_gp_grid.py", ""]
        for l in raw.splitlines():
            if keep.search(l) and "not_issued" not in l:
                txt.append("-----" if re.search(r"k_(gp|hash|tree)_", l) and "void" in l else "")
                txt.append(l.rstrip())
    if txt:
        open(os.path.join(ROOT, "profiles", f"{TAG}_ncu_gp_kernels.txt"), "w").write("\n".join(t for t in txt if t != "") + "\n")
    print("profiles written:", {k: (v[0], round(v[1] / 1e3, 1)) for k, v in per_cls.items()})


if __name__ == "__main__":
    main()
