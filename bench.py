#!/usr/bin/env python
"""bench.py — accessibility nt/s of the `db` hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N ... bench.py --gpus N ...          (one rank per GPU, launched by the driver)

A *step* is one pass of the hot path (inside + outside + accessibility, everything the reference's
`Raccess::Run` does) over config 1 of BASELINE.json IN FULL (cfg2 of SURVEY §8d: 100,000 GENCODE-like
transcripts, lognormal lengths 200-5,000 nt, 1.87e8 nt, GC 0.45, W=70, delta=5).  With N ranks the ONE
fixed dataset is split by the product's length-balanced partitioner (`priblast_b200.distributed.lpt_shard`,
the rule of csrc/host/db_format.cpp `lpt_partition`): strong scaling, no data-path collective (sequences
are independent); a step's time is the slowest rank's.  `value` is timed on the device with inputs already
resident in HBM; `e2e` is the same dataset through the public C-ABI call (`Raccess.run_batch` ->
prib_acc_run) with host buffers, H2D and D2H inside the timed region; `parity` is the deviation of the fast
engine from the reference's arithmetic (GPU exact engine, bit-pinned to the reference by the tests) on a
strided sample of the dataset, outside the timed region.

`--impl reference` times the reference's own CPU implementation (oracle/_ref, the unmodified raccess.cpp
compiled with OpenMP, all host threads) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step computed for a fixed, seeded sample of the dataset's
transcripts (the same sample whatever the number of ranks), so that two builds can be compared output for
output: DIR/acc.npy and DIR/cond.npy (float32, the (acc, cond) vectors of the sampled transcripts concatenated
in index order), DIR/transcript_index.npy (float64, the sampled transcripts' indices in the dataset) and
DIR/lengths.npy (float64, their lengths, which split acc and cond per transcript).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_SPAN = 70
DELTA = 5
N_TRANSCRIPTS = 100_000       # cfg2 in full (BASELINE.json configs[1]); --transcripts N takes the first N of the stream
WORKLOAD = ("cfg2: GENCODE-like synthetic transcripts, length=clip(round(LogNormal(ln1500,0.75)),200,5000), "
            "GC=0.45, W=70, delta=5")
# --dump-outputs sample: at most 1,024 transcripts of at most 5,000 nt, i.e. <= 41 MB of float32 (acc + cond)
DUMP_TRANSCRIPTS = 1024
DUMP_SEED = 0


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def work_per_nt(key="cfg2_W70"):
    with open(os.path.join(ROOT, "priblast_b200", "data", "work_per_nt.json")) as f:
        return json.load(f)[key]


def dataset(n: int):
    from priblast_b200 import workloads
    return workloads.cfg2(first=n)


def rank_shard(seqs, rank: int, world: int):
    """This rank's part of the one fixed dataset: the product's LPT partitioner (no collective: every rank derives
    the same deterministic split from the lengths)."""
    from priblast_b200.distributed import lpt_shard
    import numpy as np
    if world == 1:
        return list(seqs), np.arange(len(seqs))
    ids = lpt_shard([len(s) for s in seqs], world)[rank]
    return [seqs[k] for k in ids], ids


def dump_sample(n: int):
    """Sorted indices of the transcripts whose outputs --dump-outputs writes: fixed by DUMP_SEED and n alone."""
    import numpy as np
    rng = np.random.default_rng(DUMP_SEED)
    return np.sort(rng.choice(n, size=min(n, DUMP_TRANSCRIPTS), replace=False))


def write_dump(out_dir: str, ids, outputs: dict) -> None:
    """outputs: transcript index -> (acc, cond) of that transcript."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, name in enumerate(("acc", "cond")):
        arr = np.concatenate([np.asarray(outputs[int(g)][k], np.float32) for g in ids])
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)
    np.save(os.path.join(out_dir, "transcript_index.npy"), np.asarray(ids, np.float64))
    np.save(os.path.join(out_dir, "lengths.npy"), np.array([len(outputs[int(g)][0]) for g in ids], np.float64))


# ------------------------------------------------------------------------------------------------
# reference CPU arm / cpu_baseline
# ------------------------------------------------------------------------------------------------
def cpu_sample(seqs, cores: int, seconds: float = 15.0):
    """A bounded sample of the step's batch: about `seconds` of work for `cores` threads at the
    surveyed ~1.6 k nt/s/core; at least one sequence per core so every thread has work."""
    budget = 1600.0 * cores * seconds
    mean_len = max(1.0, sum(len(s) for s in seqs) / max(len(seqs), 1))
    want = int(min(len(seqs), max(cores, budget / mean_len)))
    # stride through the batch so the length mix of the sample matches the batch
    stride = max(1, len(seqs) // max(want, 1))
    take = list(seqs[::stride][:want])
    return take, sum(len(s) for s in take)


def run_cpu_reference(seqs, threads: int):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import OracleLib, RefLib
    if RefLib.available(fast=True):
        lib, kind = RefLib(fast=True), "reference"
    else:
        lib, kind = OracleLib(), "port"
    order = sorted(range(len(seqs)), key=lambda k: -len(seqs[k]))  # longest first, utils.cpp:53-60
    t0 = time.perf_counter()
    _, used = lib.run_batch([seqs[k] for k in order], W_SPAN, DELTA, nthreads=threads)
    dt = time.perf_counter() - t0
    return dt, used, kind


def reference_arm(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    cores = host_cores()
    seqs = dataset(min(args.transcripts, 4096))  # the head of the same stream: the sample is strided through it
    sample, nt = cpu_sample(seqs, cores, seconds=max(4.0, 40.0 / max(args.steps + args.warmup, 1)))
    times, used, kind = [], cores, "port"
    for it in range(args.warmup + args.steps):
        dt, used, kind = run_cpu_reference(sample, cores)
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = nt / (ms / 1e3)
    sample_desc = (f"{len(sample)} transcripts / {nt} nt strided from the first {len(seqs)} transcripts of the "
                   f"{args.transcripts}-transcript dataset; unmodified raccess.cpp, g++ -O3 -march=x86-64-v3 -fopenmp "
                   "(the reference Makefile adds -march=native -flto)")
    line = {
        "impl": "reference", "metric": "db-step accessibility throughput", "value": value, "unit": "nt/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "transcripts": args.transcripts, "sample": sample_desc, "span": W_SPAN,
                   "delta": DELTA},
        "cpu_baseline": {"value": value, "unit": "nt/s", "cores": used, "kind": kind, "sample": sample_desc},
        "e2e": {"value": value, "unit": "nt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, pw = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.rows:
            if t < t0 or t > t1 + 0.3:
                continue
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
                pw.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def ours(args, rank: int, local_rank: int, world: int) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from priblast_b200 import Raccess, _capi, packed_layout

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    result_fd = 1
    if world > 1:
        # NCCL's own log (communicator, nranks, transport) is NOT muted; it prints to stdout, which must carry exactly
        # one JSON line, so everything written to fd 1 from here on is sent to stderr and the JSON line goes out
        # through a duplicate of the real stdout.
        os.environ.setdefault("NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        sys.stdout.flush()
        result_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        print(f"[bench] NCCL communicator up: rank {rank} of nranks {dist.get_world_size()} on cuda:{local_rank} "
              f"(timing all-reduce only; the data path has no collective)", file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    all_seqs = dataset(args.transcripts)
    seqs, my_ids = rank_shard(all_seqs, rank, world)
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    nt_rank = int(lens.sum())
    nt_all = float(sum(len(s) for s in all_seqs))

    r = Raccess(W_SPAN, DELTA, device=local_rank)
    # a real (non-default) torch stream: handle 0 would mean "the context's own stream" to the library, and
    # torch events on the legacy default stream would not bracket kernels launched elsewhere
    stream = torch.cuda.Stream(device=local_rank)
    assert stream.cuda_stream != 0
    r.set_stream(stream.cuda_stream)

    # -- device-resident timing: stage once, then K x compute ----------------------------------------
    r.stage(seqs)
    for _ in range(max(args.warmup, 3)):
        r.compute()
    r.sync()
    c0 = r.counters()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_wall0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        r.compute()
    e1.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    r.sync()
    c1 = r.counters()
    if args.dump_outputs:
        # what the last timed step left on the device, fetched outside the timed region
        res = r.fetch()
        pos = {int(g): j for j, g in enumerate(my_ids)}
        dump_ids = dump_sample(len(all_seqs))
        mine = {int(g): tuple(np.array(x) for x in res[pos[int(g)]]) for g in dump_ids if int(g) in pos}
        del res
        parts = [mine]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, mine)
        if rank == 0:
            write_dump(args.dump_outputs, dump_ids, {g: v for part in parts for g, v in part.items()})
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    ms_step = ms_total / args.steps
    ms_step_max = max_over_ranks(ms_step)
    value = nt_all / (ms_step_max / 1e3)
    launches = int(c1["kernel_launches"] - c0["kernel_launches"])
    batches_per_step = (c1["batches"] - c0["batches"]) / args.steps
    phases = {k: (c1["phase_ms"][k] - c0["phase_ms"][k]) / args.steps for k in c1["phase_ms"]}

    # -- end to end through the public API with host buffers (the whole shard in ONE call) ------------
    acc_off, cond_off, total = packed_layout(lens)
    out = torch.empty(max(total, 1), dtype=torch.float32).pin_memory().numpy()
    r.run_batch(seqs, out=out)  # warm (page-locked arenas of the library)
    e2e_steps = args.steps
    c2 = r.counters()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r.run_batch(seqs, out=out)
    torch.cuda.synchronize()
    dt = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    c3 = r.counters()
    e2e_value = nt_all / dt
    h2d = int(sum_over_ranks((c3["h2d_bytes"] - c2["h2d_bytes"]) / e2e_steps))
    d2h = int(sum_over_ranks((c3["d2h_bytes"] - c2["d2h_bytes"]) / e2e_steps))
    checksum = sum_over_ranks(float(np.float64(out[:total]).sum()))
    reruns = int(sum_over_ranks(float(c1["fp64_rerun_sequences"] - c0["fp64_rerun_sequences"])) / args.steps)
    used_state = c1["dp_state_bytes_used"]
    r.close()

    if rank == 0:
        # -- parity of the fast engine against the reference's arithmetic (exact engine), outside the timed region
        stride = max(1, len(seqs) // 48)
        sample = seqs[::stride][:48]
        res = AccView(out, acc_off, cond_off, lens)
        with Raccess(W_SPAN, DELTA, device=local_rank, mode=2, max_batch_bytes=24 << 30) as rx:
            exact = rx.run_batch(sample)
        err, ref = [], []
        for j, (ea, ec) in enumerate(exact):
            fa, fc = res[j * stride]
            err.append(np.abs(np.float64(fa) - ea))
            err.append(np.abs(np.float64(fc) - ec))
            ref.append(np.abs(np.float64(ea)))
            ref.append(np.abs(np.float64(ec)))
        err, ref = np.concatenate(err), np.concatenate(ref)
        nz = ref > 1e-3
        parity = {"config": f"{len(sample)} transcripts strided from rank 0's shard, fast engine (this run's output) vs "
                            "exact engine (mode 2 = the reference's float-table log-sums on the GPU, bit-identical to "
                            "the reference in tests/test_gpu_exact.py)",
                  "unit": "kcal/mol", "n": int(err.size), "max_abs": float(err.max()), "mean_abs": float(err.mean()),
                  "max_rel": float((err[nz] / ref[nz]).max()), "tolerance_max_abs": 1e-4, "tolerance_mean_abs": 5e-6}

        # -- roofline of the dominant kernel (SURVEY §8d: SFU-issue bound on algorithmic terms) --------
        lib = _capi.load()
        import ctypes
        mufu, ffma, dfma = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        _capi.check(lib.prib_peak_probe(local_rank, ctypes.byref(mufu), ctypes.byref(ffma), ctypes.byref(dfma)))
        wk = work_per_nt()
        dom = max((k for k in phases if k != "memset"), key=lambda k: phases[k])
        # whole-step algorithmic SFU work / whole-step device time (all kernels of the step together
        # evaluate the recurrences; per-phase shares are given beside it); rank 0's shard over rank 0's time
        sfu_ops = wk["sfu_ops_per_nt"] * nt_rank
        achieved = sfu_ops / (ms_step * 1e-3) / 1e9
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        # the dominant kernel on its own: its share of the algorithmic terms over its own device time; one launch
        # per device batch (the dataset takes several: the DP state of a batch fills the HBM budget)
        phase_terms = {"inside": wk.get("terms_inside_per_nt"), "outside": wk.get("terms_outside_per_nt"),
                       "biloop_left": None, "biloop_right": None}
        dom_kernel = {"inside": "k_inside_tile", "outside": "k_outside_tile", "biloop_left": "k_biloop_tile<LEFT>",
                      "biloop_right": "k_biloop_tile<RIGHT>"}.get(dom, dom)
        nt_launch = nt_rank / max(batches_per_step, 1)
        dom_obj = {"phase": dom, "kernel": dom_kernel, "launches_per_step": batches_per_step,
                   "ms_per_launch": phases[dom] / max(batches_per_step, 1), "nt_per_launch": nt_launch}
        if phase_terms.get(dom):
            # 6 band variables of this pass = 6 (W-1) reduction outputs per nt
            ops = (phase_terms[dom] + 6 * (W_SPAN - 1)) * nt_rank
            dom_obj.update({"sfu_ops_per_nt": phase_terms[dom] + 6 * (W_SPAN - 1),
                            "achieved": ops / (phases[dom] * 1e-3) / 1e9,
                            "frac": ops / (phases[dom] * 1e-3) / 1e9 / mufu.value})
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r2", "traffic.json")) as f:
                tj = json.load(f)
            if tj["kernel"].startswith(dom_kernel):  # measured bytes per nt of that kernel (one ncu --set full capture)
                traffic = (tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]) / tj["nt_per_launch"] * nt_launch
        except Exception:
            pass
        roofline = {
            "bound": "sfu", "achieved": achieved, "peak": mufu.value, "unit": "Gop/s", "frac": achieved / mufu.value,
            "traffic": traffic, "dominant_kernel": dom_obj,
            "definition": "algorithmic terms x 1 EX2 + reduction outputs x 1 LG2 per second (SURVEY 8d) over the "
                          "measured MUFU ex2.approx issue peak of this GPU (prib_peak_probe, same run); the kernels "
                          "work in the linear domain and issue no MUFU: this is the survey's accounting yardstick, "
                          "not a pipe utilisation (profiles/r2 holds the pipe counters)",
            "sfu_ops_per_nt": wk["sfu_ops_per_nt"], "terms_per_nt": wk["terms_per_nt"],
            "fp32_frac": (6 * wk["terms_per_nt"] * nt_rank / (ms_step * 1e-3) / 1e9) / ffma.value,
            "peaks_measured_gops": {"mufu_ex2": mufu.value, "ffma": ffma.value, "dfma": dfma.value},
            "dominant_phase": dom, "phase_ms_per_step": phases,
            "hbm": {"peak_gbs": hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                    "algorithmic_bytes_per_nt": 9.0,
                    "achieved_gbs": 9.0 * nt_rank / (ms_step * 1e-3) / 1e9},
        }
        # -- CPU baseline beside it (N=1 only) ---------------------------------------------------------
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = host_cores()
            sample_c, nt_s = cpu_sample(all_seqs[:4096], cores, seconds=15.0)
            dtc, used, kind = run_cpu_reference(sample_c, cores)
            cpu = {"value": nt_s / dtc, "unit": "nt/s", "cores": used, "kind": kind,
                   "sample": f"{len(sample_c)} transcripts / {nt_s} nt strided from the first 4,096 transcripts of the "
                             f"dataset, {dtc:.1f} s; unmodified raccess.cpp, g++ -O3 -march=x86-64-v3 -fopenmp (the "
                             "reference Makefile adds -march=native -flto)"}
        line = {
            "metric": "db-step accessibility throughput", "value": value, "unit": "nt/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step_max,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "transcripts": len(all_seqs), "nt": int(nt_all),
                       "arithmetic": "band DP in f32 (span-scaled, range-guarded, f64 re-run of flagged sequences: "
                       + str(reruns) + " per step); outer arrays and final sums in f64",
                       "nt_rank0": nt_rank, "device_batches_per_step_rank0": batches_per_step,
                       "span": W_SPAN, "delta": DELTA,
                       "l2_policy": f"no flush needed: every device batch rewrites {used_state / 2**30:.1f} GiB of DP state "
                                    "(>> 126 MB L2)",
                       "parallelism": f"one fixed dataset, LPT-split (priblast_b200.distributed.lpt_shard) over {world} "
                                      "rank(s), no collective"},
            "e2e": {"value": e2e_value, "unit": "nt/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "seconds_per_step": dt, "checksum": checksum,
                    "what": "the whole dataset through Raccess.run_batch -> prib_acc_run per rank, host buffers in, "
                            "page-locked host image out; slowest rank"},
            "parity": parity,
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        }
        sys.stdout.flush()
        os.write(result_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


class AccView:
    """(acc, cond) views of sequence k in a packed output image."""

    def __init__(self, out, acc_off, cond_off, lens):
        self.out, self.a, self.c, self.l = out, acc_off, cond_off, lens

    def __getitem__(self, k):
        a, c, l = int(self.a[k]), int(self.c[k]), int(self.l[k])
        return self.out[a:a + l], self.out[c:c + l]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--transcripts", type=int, default=N_TRANSCRIPTS,
                    help="take the first N transcripts of the cfg2 stream (default: the whole config, 100,000)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs for a fixed sample of transcripts to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
