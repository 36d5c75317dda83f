"""bench.py -- distinct states/sec of the BFS frontier-expansion path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one complete explicit-state BFS (Init -> empty frontier) of the headline model:
Kip320 bound to KafkaReplication.tla, 3 brokers, LogSize ("MaxLogLen") 4, MaxRecords 4, MaxLeaderEpoch 3
(models/Kip320_R4.cfg: 340,433,359 distinct states, depth 42).
The input is the .cfg; there is no RNG.  The result of every step (distinct, generated, depth,
per-level widths) is compared with the committed golden before a number is printed.

  value        total distinct states / CUDA-event time of the level loop, state store and hash set
               already allocated in HBM, max over ranks
  e2e          the same through the C-ABI call a TLC-side caller makes (kmc_run + kmc_stats +
               kmc_level_widths), wall clock: includes the hash-set reset, the host->device copy of the
               initial states and the per-level device->host counter reads
  roofline     dominant kernel by time, live CUDA-event launch durations (engine stream)
  e2e_cold     what a tlc2 user pays for a NEW .cfg: parse + lower (measured on the build host, model.json) +
               nvcc of the lowered model (timed live, on this box) + library load, kmc_create and the first kmc_run
  cpu_baseline baseline/cpu_bfs.cpp: the SAME lowered Next / invariants compiled for the host (-O3 -march=native),
               packed states, lock-free 64-bit fingerprint table, persistent worker pool, per-thread output
               buffers, all host threads -- a full BFS of the same .cfg when it fits the time budget (kind "port":
               TLC itself cannot run here, no JVM).  Oracle B stays what it is: the checker.

--impl reference times that CPU path alone (rank 0 only).

--dump-outputs DIR writes what the last timed step computed (single GPU), for comparing two builds:
  counts.npy         float64 [distinct, generated, depth, queue, deadlocks, complete]
  levels.npy         float64 per-level widths (distinct states first reached at each BFS level)
  states_sample.npy  float64 [rows, 2*words]: the reachable states whose salted hash falls in a fixed residue
                     class (about 2^18 of them), each 64-bit word split into its high and low 32 bits, rows
                     sorted -- a sample chosen by content, so it does not depend on the order of the state store
Nothing is written to the source tree: run-time builds (the cold-start nvcc output, the CPU arm's library) go to a
temporary directory removed at exit.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_MODEL = "kip320_3x4_r4e3"
METRIC = "distinct states/sec"
SAMPLE_SALT = 0x5EED_0F_C0FFEE          # fixed seed of the state sample written by --dump-outputs
SAMPLE_ROWS_LOG2 = 18                  # about 2^18 sampled states: 2^18 rows * 2 words * 2 halves * 8 B = 8 MB for W = 2

_SCRATCH = None


def scratch_dir() -> str:
    """A private temporary directory for what the benchmark compiles at run time; the tree may be read-only."""
    global _SCRATCH
    if _SCRATCH is None:
        _SCRATCH = tempfile.mkdtemp(prefix="kspec-bench-")
        atexit.register(shutil.rmtree, _SCRATCH, True)
    return _SCRATCH


def load_json(path):
    with open(path) as f:
        return json.load(f)


def _mix64(x: np.ndarray) -> np.ndarray:
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)."""
    x = x ^ (x >> np.uint64(30))
    x = x * np.uint64(0xBF58476D1CE4E5B9)
    x = x ^ (x >> np.uint64(27))
    x = x * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def sample_states(ck, distinct: int, chunk_rows: int = 1 << 24) -> np.ndarray:
    """The reachable states whose salted content hash is 0 modulo max(1, distinct >> SAMPLE_ROWS_LOG2), sorted;
    returned as float64 with every uint64 word split into (high 32 bits, low 32 bits), which float64 holds exactly."""
    modulus = np.uint64(max(1, distinct >> SAMPLE_ROWS_LOG2))
    picked = []
    for first in range(0, distinct, chunk_rows):
        rows = ck.copy_states(first, min(chunk_rows, distinct - first))
        h = np.full(len(rows), SAMPLE_SALT, dtype=np.uint64)
        for k in range(rows.shape[1]):
            h = _mix64(h ^ rows[:, k])
        picked.append(rows[h % modulus == 0])
    rows = np.concatenate(picked) if picked else np.zeros((0, ck.words), dtype=np.uint64)
    rows = rows[np.lexsort(rows.T[::-1])] if len(rows) else rows
    halves = np.stack([rows >> np.uint64(32), rows & np.uint64(0xFFFFFFFF)], axis=2).reshape(len(rows), -1)
    return halves.astype(np.float64)


def dump_outputs(out_dir: str, ck, res) -> None:
    """Writes the last timed step's result (see the module docstring) as float64 .npy files."""
    os.makedirs(out_dir, exist_ok=True)
    counts = [res.distinct, res.generated, res.depth, res.queue, res.deadlocks, int(res.complete)]
    np.save(os.path.join(out_dir, "counts.npy"), np.array(counts, dtype=np.float64))
    np.save(os.path.join(out_dir, "levels.npy"), np.array(res.levels, dtype=np.float64))
    np.save(os.path.join(out_dir, "states_sample.npy"), sample_states(ck, res.distinct))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = load_json(p)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def nvlink_counters(gpu_index: int):
    """Cumulative NVLink data counters of one GPU (sum over its links), in bytes, from `nvidia-smi nvlink -gt d`
    ("Data Tx: N KiB" / "Data Rx: N KiB" per link); None when the tool, the option or the links are not there."""
    import re
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(gpu_index)], capture_output=True, text=True,
                             timeout=20).stdout
    except (OSError, subprocess.SubprocessError):
        return None
    tx = [int(x) for x in re.findall(r"Data Tx:\s*(\d+)\s*KiB", out)]
    rx = [int(x) for x in re.findall(r"Data Rx:\s*(\d+)\s*KiB", out)]
    if not tx or not rx:
        return None
    return {"tx": 1024 * sum(tx), "rx": 1024 * sum(rx), "links": len(tx)}


def golden_for(model: str):
    g = load_json(os.path.join(ROOT, "tests", "golden", "goldens.json"))
    return g.get(model)


def check_result(model, distinct, generated, depth, levels, deadlocks):
    g = golden_for(model)
    if g is None:
        return "no golden committed for this model"
    got = (distinct, generated, depth, deadlocks, levels)
    want = (g["distinct"], g["generated"], g["depth"], g["deadlocks"], g["levels"])
    if got != want:
        raise SystemExit(f"PARITY FAILURE on {model}: got {got[:4]}, golden {want[:4]}")
    return "bit-exact vs tests/golden/goldens.json (" + "+".join(g["sources"]) + ")"


def cpu_run(model: str, threads: int = 0, budget_s: float = 25.0, table_log2: int = 0):
    """One run of the CPU arm (baseline/cpu_bfs.cpp).  A short bounded probe gives the rate; if the full BFS is
    expected to fit `budget_s` it is run in full (same_config true, result checked against the golden), else the
    run is bounded to about budget_s of work."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import cpu_bfs
    cores = os.cpu_count() or 1
    threads = threads or cores
    g = golden_for(model)
    total = g["distinct"] if g else 0
    if not table_log2:
        table_log2 = 20
        while (1 << table_log2) < 2.5 * max(total, 1 << 18):
            table_log2 += 1
    probe = cpu_bfs.run(model, threads, min(table_log2, 26), stop_after_states=2_000_000, out_dir=scratch_dir())
    rate = probe["distinct"] / max(probe["seconds"], 1e-9)
    full = bool(total) and (probe["complete"] or total / rate <= budget_s)
    if probe["complete"]:
        r = probe
    else:
        r = cpu_bfs.run(model, threads, table_log2, stop_after_states=0 if full else int(rate * budget_s),
                        out_dir=scratch_dir())
    if r["fail"]:
        raise SystemExit(f"cpu baseline failed on {model}: code {r['fail']}")
    if r["complete"] and g:
        got = (r["distinct"], r["generated"], r["depth"], r["deadlocks"], r["levels"])
        want = (g["distinct"], g["generated"], g["depth"], g["deadlocks"], g["levels"])
        if got != want:
            raise SystemExit(f"CPU baseline disagrees with the golden on {model}: {got[:4]} vs {want[:4]}")
    what = "full BFS" if r["complete"] else f"first {r['distinct']} distinct states ({r['depth']} levels)"
    return {"value": r["distinct"] / max(r["seconds"], 1e-9), "unit": "states/s", "cores": threads, "kind": "port",
            "same_config": bool(r["complete"]), "seconds": r["seconds"], "distinct": r["distinct"],
            "sample": f"baseline/cpu_bfs.cpp (the lowered Next of {model} compiled for the host, packed states, lock-free "
                      f"64-bit fingerprint table, {threads} of {cores} host threads): {what} in {r['seconds']:.2f} s; "
                      f"TLC itself unavailable (no JVM)"}


def cpu_scaling(model: str):
    """Bounded samples at 1 and 16 threads (the scaling reference next to the all-threads number)."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import cpu_bfs
    out = {}
    for t in (1, 16):
        if t > (os.cpu_count() or 1):
            continue
        r = cpu_bfs.run(model, t, 25, stop_after_states=1_500_000 * t, out_dir=scratch_dir())
        out[str(t)] = round(r["distinct"] / max(r["seconds"], 1e-9))
    return out


def config_for(model: str, extra: dict | None = None) -> dict:
    reg = load_json(os.path.join(ROOT, "models", "MODELS.json"))[model]
    params = (reg.get("kso") or [None, None])[1]
    what = (f"KafkaReplication.tla {params[0]} brokers LogSize {params[1]} MaxRecords {params[2]} MaxLeaderEpoch {params[3]}"
            if params and len(params) == 4 else f"params {params}")
    c = {"workload": f"{reg['module']} ({reg['cfg']}): full BFS, {what}",
         "model": model, "l2": "inputs larger than L2: hash set and state store are GBs and the set is reset every step"}
    if extra:
        c.update(extra)
    return c


def run_reference(args):
    """The CPU arm alone (rank 0): every step is one run of baseline/cpu_bfs.cpp on all host threads -- the full
    BFS of the same .cfg when a run fits ~40 s, else a bounded prefix (same_config false)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # a CPU run has no clocks to ramp and no caches worth warming across 10^8-state searches: one warm-up run at most,
    # and a per-step budget that keeps the whole arm (probe + steps + the two scaling samples) to a few minutes
    # The first timed step is the anchor: up to 75 s, i.e. the FULL BFS of the same cfg whenever the host manages it in
    # that time (same_config true, result checked against the golden); the remaining steps are bounded prefixes sized
    # so that the whole arm stays within a few minutes for any --steps.
    warm = 0
    vals = []
    for i in range(args.steps):
        budget = 75.0 if i == 0 else max(4.0, min(25.0, 90.0 / max(1, args.steps - 1)))
        vals.append(cpu_run(args.model, budget_s=budget))
    total_states = sum(v["distinct"] for v in vals)
    total_s = sum(v["seconds"] for v in vals)
    value = total_states / total_s
    last = vals[0]                  # the anchor step describes the arm (same_config, sample text)
    line = {"metric": METRIC, "value": value, "unit": "states/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * total_s / max(1, args.steps), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic (the .cfg is the input)",
            "impl": "reference", "config": config_for(args.model, {"same_config": last["same_config"]}),
            "cpu_baseline": {"value": value, "unit": "states/s", "cores": last["cores"], "kind": "port",
                             "sample": last["sample"] + f"; then {args.steps - 1} bounded prefixes of the same search",
                             "same_config": last["same_config"], "anchor_step_states_per_s": last["value"],
                             "thread_scaling_states_per_s": cpu_scaling(args.model)},
            "e2e": {"value": value, "unit": "states/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def cold_start(model: str, opts: dict):
    """A new .cfg, end to end: (parse + lower, measured when the model was lowered on the build host; the .tla
    sources are not on this box) + nvcc of the lowered header, live + dlopen/kmc_create + the first kmc_run."""
    from kafka_specification_b200 import build as B
    from kafka_specification_b200.runtime import Checker
    meta = load_json(os.path.join(B.model_dir(model), "model.json"))
    so = os.path.join(scratch_dir(), f"libkmc_{model}.cold.so")
    t0 = time.perf_counter()
    B.compile_model_to(model, so)
    t1 = time.perf_counter()
    ck = Checker(model, model_lib=so, **opts)
    r = ck.run()
    t2 = time.perf_counter()
    ck.close()
    lower_s = float(meta.get("lower_seconds", 0.0))
    total = lower_s + (t2 - t0)
    return {"seconds": total, "lower_s": lower_s, "nvcc_s": t1 - t0, "load_create_run_s": t2 - t1,
            "value": r.distinct / total, "unit": "states/s",
            "note": "lower_s measured on the build host (the .tla sources are not shipped to the GPU box); the rest live"}


def run_single(args):
    import torch
    from kafka_specification_b200.runtime import Checker
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    opts = {"device": dev}
    if args.table_log2:
        opts["table_log2"] = args.table_log2
    if args.max_states:
        opts["max_states"] = args.max_states
    ck = Checker(args.model, **opts)
    for _ in range(args.warmup):
        ck.run()
    sampler = ClockSampler(dev)
    sampler.start()
    torch.cuda.synchronize()
    gpu_ms, e2e_ms, launches = [], [], 0
    exp_ms = ins_ms = inv_ms = 0.0
    n_exp = n_ins = n_inv = 0
    res = None
    t_bracket = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter()
        res = ck.run()                         # kmc_run + kmc_stats + kmc_level_widths + kmc_violation
        e2e_ms.append(1000.0 * (time.perf_counter() - t0))
        st = res.stats
        gpu_ms.append(st["gpu_ms_total"])
        launches += st["launches_expand"] + st["launches_insert"] + st["launches_other"]
        exp_ms += st["gpu_ms_expand"]
        ins_ms += st["gpu_ms_insert"]
        inv_ms += st["gpu_ms_invariant"]
        n_exp += st["launches_expand"]
        n_ins += st["launches_insert"]
        n_inv += st["launches_other"]
    torch.cuda.synchronize()
    bracket_ms = 1000.0 * (time.perf_counter() - t_bracket)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ck, res)
    parity = check_result(args.model, res.distinct, res.generated, res.depth, res.levels, res.deadlocks)
    if res.violation is not None or not res.complete:
        raise SystemExit(f"bench: unexpected verdict {res.violation}")
    W = ck.words
    S = 8 * W
    X, G, N = res.distinct, res.generated, res.distinct
    steps = args.steps
    value = steps * N / (sum(gpu_ms) / 1000.0)
    e2e = steps * N / (sum(e2e_ms) / 1000.0)
    peak, peak_src = measured_peaks()
    # algorithmic bytes per BFS (SURVEY 8d): expand reads X*S and writes G*(S+8); the hash probe
    # reads G candidate rows' buckets (32 B each) and writes N*8 (slot) -- plus N*(S+8) store/parent
    exp_bytes = X * S + G * (S + 8)
    ins_bytes = G * 32 + N * 8
    inv_bytes = N * (S + 8)
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        traffic = load_json(tp).get(args.model, {})

    def roof(kernel, bytes_per_bfs, total_ms, n_launch):
        sec = total_ms / 1000.0
        ach = steps * bytes_per_bfs / sec / 1e9 if sec > 0 else 0.0
        ratio = (traffic.get(kernel) or {}).get("traffic_over_algorithmic")
        per_launch = steps * bytes_per_bfs / max(1, n_launch)
        return {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": (ratio * per_launch) if ratio else None, "traffic_over_algorithmic": ratio,
                "peak_source": peak_src,
                "avg_launch_ms": total_ms / max(1, n_launch), "launches": n_launch,
                "algorithmic_bytes_per_launch": steps * bytes_per_bfs / max(1, n_launch),
                "share_of_gpu_time": total_ms / max(1e-9, sum(gpu_ms))}

    r_exp = roof("k_expand", exp_bytes, exp_ms, n_exp)
    r_ins = roof("k_insert", ins_bytes, ins_ms, n_ins)
    # secondary denominator for the hash-probe kernel: measured random 32 B-sector gather rate on a table
    # of the same size (tools/gather_bench.cu -> profiles/gather_peak.json)
    gp = os.path.join(ROOT, "profiles", "gather_peak.json")
    if os.path.exists(gp) and ins_ms > 0:
        want = res.stats["table_slots"] * (res.stats.get("slot_bytes") or 8)
        pts = load_json(gp)["results"]
        best = min(pts, key=lambda r: abs(r["table_bytes"] - want))
        probes_per_s = steps * res.stats["probes"] / (ins_ms / 1000.0)
        r_ins["random_gather_peak_probes_per_s"] = best["probes_per_s"]
        r_ins["probes_per_s"] = probes_per_s
        r_ins["frac_of_random_gather_peak"] = probes_per_s / best["probes_per_s"]
    r_inv = roof("k_invariants", inv_bytes, inv_ms, n_inv)
    ranked = sorted([r_exp, r_ins, r_inv], key=lambda r: -r["share_of_gpu_time"])
    dominant, other = ranked[0], ranked[1:]
    # the auxiliary legs must never cost the headline line: a failure there is reported in place of the number
    cpu = cold = None
    if not args.no_cpu_baseline:
        try:
            cpu = cpu_run(args.model)
        except BaseException as e:                       # (cpu_run raises SystemExit on a parity failure)
            cpu = {"value": None, "unit": "states/s", "cores": os.cpu_count(), "kind": "port", "same_config": False,
                   "sample": f"cpu baseline failed: {e!r}"[:300]}
    if not args.no_cold:
        try:
            cold = cold_start(args.model, opts)
        except BaseException as e:
            cold = {"seconds": None, "error": repr(e)[:300]}
    info = ck.info
    depth = res.depth
    line = {
        "metric": METRIC, "value": value, "unit": "states/s", "n_gpus": 1, "steps": steps, "warmup": args.warmup,
        "ms_per_step": sum(gpu_ms) / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic (the .cfg is the input; no RNG)",
        "config": config_for(args.model, {"distinct": N, "generated": G, "depth": depth, "state_words": W,
                                          "table_slots": res.stats["table_slots"], "parity": parity,
                                          "exact_fingerprints": bool(info.exact)}),
        "roofline": dominant, "roofline_other": other,
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")} if cpu else None,
        "e2e_cold": cold,
        "e2e": {"value": e2e, "unit": "states/s", "ms_per_step": sum(e2e_ms) / steps,
                "h2d_bytes_per_step": info.num_init * (W + 1) * 8 + 8 * 16 + (depth + 1) * 64,
                "d2h_bytes_per_step": (depth + 1) * (17 + 64) * 8 + 18 * 8 + depth * 8},
        "bracket_ms_per_step": bracket_ms / steps,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    ck.close()
    return 0


def run_sharded(args):
    import torch
    import torch.distributed as dist
    from kafka_specification_b200.sharded import CudaShardEngine, ShardedChecker
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    opts = {}
    if args.table_log2:
        opts["table_log2"] = args.table_log2
    if args.max_states:
        opts["max_states"] = args.max_states
    if args.no_p2p:
        opts["p2p"] = False
    eng = CudaShardEngine(args.model, rank, world, local, **opts)
    drv = ShardedChecker(eng)
    g = golden_for(args.model)
    sync_note = None

    def agreed_run():
        """One run on every rank; all ranks learn whether it succeeded everywhere and matched the golden."""
        r, err = None, None
        try:
            r = drv.run()
            if g and (r.distinct, r.generated, r.depth, r.levels) != (g["distinct"], g["generated"], g["depth"], g["levels"]):
                err = f"result differs from the golden: {(r.distinct, r.generated, r.depth)}"
        except Exception as ex:                       # KmcError (incl. KMC_E_PEER_TIMEOUT), RuntimeError
            err = repr(ex)[:200]
        ok = torch.tensor([0 if err else 1], dtype=torch.int64, device=eng.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return r, err, bool(ok.item())

    # The first warm-up run doubles as the acceptance run of the device-side round/level synchronisation (flags in
    # peer memory): if it fails on any rank, every rank falls back to the stream-ordered NCCL barrier per round (the
    # exchange itself stays fused) -- and the line says so.
    if args.warmup > 0 and eng.p2p and eng.device_sync:
        _, err, ok = agreed_run()
        if not ok:
            errs = [None] * world
            dist.all_gather_object(errs, err)
            sync_note = "device-side sync failed in the first warm-up run, NCCL barrier per round used instead: " + \
                        "; ".join(f"rank {i}: {e}" for i, e in enumerate(errs) if e)
            if rank == 0:
                print("[bench] " + sync_note, file=sys.stderr, flush=True)
            eng.device_sync = False
        n_warm = args.warmup - 1
    else:
        n_warm = args.warmup
    for _ in range(n_warm):
        drv.run()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dist.barrier()
    torch.cuda.synchronize()
    nvl0 = nvlink_counters(local) if rank == 0 else None
    secs, gpu_ms, launches = [], [], 0
    ins_ms = exp_ms = 0.0
    n_ins = n_exp = 0
    res = None
    for _ in range(args.steps):
        res = drv.run()                         # barrier inside; seconds = max over ranks
        secs.append(res.seconds)
        st = res.stats
        gpu_ms.append(st["gpu_ms_total"])
        launches += st["launches_expand"] + st["launches_insert"] + st["launches_other"]
        exp_ms += st["gpu_ms_expand"]
        ins_ms += st["gpu_ms_insert"]
        n_exp += st["launches_expand"]
        n_ins += st["launches_insert"]
    dist.barrier()
    torch.cuda.synchronize()
    # device time of the level loop: max over ranks of the CUDA-event total
    t = torch.tensor([sum(gpu_ms)], dtype=torch.float64, device=eng.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gpu_total_ms = float(t.item())
    lt = torch.tensor([launches], dtype=torch.int64, device=eng.device)
    dist.all_reduce(lt)
    clocks = sampler.stop() if rank == 0 else None
    nvl1 = nvlink_counters(local) if rank == 0 else None
    nvlink_measured = None
    if nvl0 and nvl1:
        nvlink_measured = {"gpu": local, "links": nvl1["links"],
                           "tx_bytes_per_step": (nvl1["tx"] - nvl0["tx"]) / max(1, args.steps),
                           "rx_bytes_per_step": (nvl1["rx"] - nvl0["rx"]) / max(1, args.steps),
                           "source": "nvidia-smi nvlink -gt d, rank 0's GPU, counters read before and after the timed steps"}
    if rank == 0:
        parity = check_result(args.model, res.distinct, res.generated, res.depth, res.levels, res.deadlocks)
        steps = args.steps
        N, G = res.distinct, res.generated
        W = eng.ck.words
        value = steps * N / (gpu_total_ms / 1000.0)
        e2e = steps * N / sum(secs)
        peak, peak_src = measured_peaks()
        ins_bytes = (G * 32 + N * 8) / world
        ach = steps * ins_bytes / (ins_ms / 1000.0) / 1e9 if ins_ms else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": "states/s", "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": gpu_total_ms / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic (the .cfg is the input; no RNG)",
            "config": config_for(args.model, {"distinct": N, "generated": G, "depth": res.depth, "state_words": W,
                                              "parity": parity, "parallelism": f"fingerprint-sharded x{world}",
                                              "exchange": "fused: expand kernel stores rows into the owners' inboxes over NVLink (CUDA IPC)"
                                              if eng.p2p else "NCCL all-to-all-v per chunk",
                                              "round_sync": ("device-side flags in peer memory, one host sync per level"
                                                             if (eng.p2p and eng.device_sync) else
                                                             "stream-ordered NCCL barrier per round, host read-back per level"),
                                              "round_sync_note": sync_note,
                                              "nvlink_bytes_per_step_est": int(G * (world - 1) / world * (W + 1) * 8),
                                              "nvlink_measured": nvlink_measured,
                                              "per_rank_distinct": res.per_rank_distinct,
                                              "exchanged_rows_per_step": res.exchanged_rows}),
            "roofline": {"kernel": "k_insert (rank 0)", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "avg_launch_ms": ins_ms / max(1, n_ins), "launches": n_ins},
            "cpu_baseline": None,
            "e2e": {"value": e2e, "unit": "states/s", "ms_per_step": 1000.0 * sum(secs) / steps,
                    "h2d_bytes_per_step": (res.depth + 1) * 64 * world, "d2h_bytes_per_step": (res.depth + 1) * 81 * 8 * world},
            "gpu_launches": int(lt.item()),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    eng.close()
    dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default=DEFAULT_MODEL)
    ap.add_argument("--table-log2", type=int, default=0)
    ap.add_argument("--max-states", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cold", action="store_true", help="skip the cold-start (nvcc + first run) measurement")
    ap.add_argument("--no-p2p", action="store_true", help="multi-GPU: NCCL all-to-all exchange instead of the fused peer-memory path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="single GPU: write the last timed step's result to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    # Sizing is configuration (like TLC's -fpmem), not derived from the answer: 2^30 set slots and room for 2^29
    # states per rank for the headline class of models; an overflow is reported (KMC_E_TABLE_FULL / STORE_FULL).
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not args.table_log2:
        args.table_log2 = 30 if world == 1 else 29
    if not args.max_states:
        args.max_states = (1 << 29) if world == 1 else (1 << 28)
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        ap.error("--dump-outputs is supported for the single-GPU run of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if world > 1:
        return run_sharded(args)
    return run_single(args)


if __name__ == "__main__":
    sys.exit(main())
