"""k minimum accessible lengths from one context against k single-length contexts (DESIGN.md §2.10).

Workload: the first 10,000 transcripts of bench.py's cfg2 stream (a 10 % sample: lognormal lengths around 1.5 kb, GC
0.45), at W = 70 and W = 150, default mode.  For k = 1, 2, 4, 8 the lengths are the first k of LENGTHS.  Every context
keeps its own DP state (max_batch_bytes = 10 GiB each, so that the twelve contexts of one span fit the card) and
writes into one page-locked output buffer (the direct-copy path of prib_acc_fetch).  Each repetition times, in
alternating order, one prib_acc_run of the k-length context and one prib_acc_run of each of the k single-length
contexts: end to end (host clock around the blocking call) and device time (the kernel_ms counter).  The ratio is
multi / sum of singles; below 1 the shared inside / outside passes pay off.

usage: python profiles/multi_length.py [--out FILE.jsonl] [--reps 3] [--transcripts 10000]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

LENGTHS = (5, 8, 10, 12, 15, 20, 25, 30)
KS = (1, 2, 4, 8)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed_run(r, seqs, out):
    k0 = r.counters()["kernel_ms"]
    t0 = time.perf_counter()
    r.run_batch(seqs, out=out)
    t1 = time.perf_counter()
    return (t1 - t0) * 1e3, r.counters()["kernel_ms"] - k0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--transcripts", type=int, default=10_000)
    ap.add_argument("--spans", default="70,150")
    a = ap.parse_args()
    from priblast_b200 import Raccess, _capi, workloads
    seqs = workloads.cfg2(first=a.transcripts)
    nt = sum(map(len, seqs))
    lib = _capi.load()
    floats = 2 * nt * max(KS)
    buf = lib.prib_host_alloc(4 * floats)
    if not buf:
        raise RuntimeError("prib_host_alloc failed")
    out = np.ctypeslib.as_array(ctypes.cast(buf, _capi.c_f32p), shape=(floats,))
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    emit({"card": card(), "transcripts": len(seqs), "nucleotides": nt, "lengths": LENGTHS, "reps": a.reps})
    budget = 10 << 30
    for W in (int(w) for w in a.spans.split(",")):
        singles = {d: Raccess(W, d, max_batch_bytes=budget) for d in LENGTHS}
        multis = {k: Raccess(W, list(LENGTHS[:k]), max_batch_bytes=budget) for k in KS}
        for r in list(singles.values()) + list(multis.values()):  # warm-up: modules, DP state, pinned arenas
            r.run_batch(seqs, out=out)
        for k in KS:
            m_e2e, m_dev, s_e2e, s_dev = [], [], [], []
            for rep in range(a.reps):
                def multi():
                    e, d = timed_run(multis[k], seqs, out)
                    m_e2e.append(e)
                    m_dev.append(d)

                def single():
                    e = d = 0.0
                    for delta in LENGTHS[:k]:
                        e1, d1 = timed_run(singles[delta], seqs, out)
                        e += e1
                        d += d1
                    s_e2e.append(e)
                    s_dev.append(d)
                order = (multi, single) if rep % 2 == 0 else (single, multi)
                for f in order:
                    f()
            med = lambda v: float(np.median(v))
            emit({"W": W, "k": k, "lengths": LENGTHS[:k],
                  "multi_e2e_ms": med(m_e2e), "singles_e2e_ms": med(s_e2e), "ratio_e2e": med(m_e2e) / med(s_e2e),
                  "multi_kernel_ms": med(m_dev), "singles_kernel_ms": med(s_dev), "ratio_kernel": med(m_dev) / med(s_dev),
                  "multi_e2e_runs": m_e2e, "singles_e2e_runs": s_e2e,
                  "phase_ms_multi_total": multis[k].counters()["phase_ms"]})
        for r in list(singles.values()) + list(multis.values()):
            r.close()
    lib.prib_host_free(buf)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
