"""Wide spans: device throughput of the wide-span FP64 engine (modes 0 / 1 above W = 200; the FP32 tile engine at
W = 200) and of the exact engine (mode 2) on the same uniform 2 kb sequences of workloads.cfg4, per W.  Rates are
nucleotides over the device time of prib_acc_compute (CUDA events, counters()["kernel_ms"]) after a warm-up call in
the same context.  Prints one JSON line per (W, engine) and a header line with the card and its power limit.
usage: wide_span.py [--n 1000] [--spans 200,201,250,400,1000] [--exact-n W:n,...] [--out file.jsonl]"""
import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def default_klog2() -> float:
    src = open(os.path.join(ROOT, "priblast_b200", "csrc", "acc_tables.h")).read()
    body = src[src.index("default_scale_wide()"):]
    return float(re.search(r"s\.klog2 = ([0-9.]+);", body).group(1))


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def measure(seqs, W, mode):
    from priblast_b200 import Raccess
    with Raccess(W, 5, mode=mode) as r:
        r.run_batch(seqs[:8])  # warm-up: module load, first allocations
        c0 = r.counters()
        r.stage(seqs)
        r.compute()
        r.sync()
        c1 = r.counters()
    nt = c1["nucleotides"] - c0["nucleotides"]
    ms = c1["kernel_ms"] - c0["kernel_ms"]
    return {"sequences": c1["sequences"] - c0["sequences"], "nt": nt, "device_ms": round(ms, 1),
            "nt_per_s": nt / (ms / 1e3), "exact_rerun_sequences": c1["exact_rerun_sequences"] - c0["exact_rerun_sequences"],
            "fp64_rerun_sequences": c1["fp64_rerun_sequences"] - c0["fp64_rerun_sequences"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--spans", default="200,201,250,400,1000")
    ap.add_argument("--exact-n", default="", help="W:n pairs: fewer sequences for the exact engine at these spans")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from priblast_b200 import workloads
    seqs = workloads.cfg4(first=a.n)
    exact_n = {int(k): int(v) for k, v in (p.split(":") for p in a.exact_n.split(",") if p)}
    klog2 = float(os.environ.get("PRIB_WIDE_KLOG2", default_klog2()))
    lines = [dict(card(), workload=f"cfg4 {a.n} x 2000 nt", delta=5, wide_klog2=klog2)]
    print(json.dumps(lines[0]), flush=True)
    for W in (int(x) for x in a.spans.split(",")):
        for engine, mode in (("tile_fp32" if W <= 200 else "wide_fp64", 0), ("exact", 2)):
            n = exact_n.get(W, a.n) if mode == 2 else a.n
            row = dict(W=W, engine=engine, **measure(seqs[:n], W, mode))
            if mode == 0 and W > 200:
                row["kappa"] = f"2^-{klog2}"
            lines.append(row)
            print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
