"""bench.py's single-GPU leg with the GPU stubbed out: the JSON line's contract (keys the driver reads, the roofline /
cpu_baseline / e2e objects) is assembled by ordinary Python that a typo could break without any test noticing until
the round-end run.  The stub only stands in for kmc_run's numbers; nothing here is a measurement."""
import json
import os
import sys
import types

import pytest

from conftest import ROOT


class _FakeResult:
    def __init__(self, g, words):
        self.distinct, self.generated, self.depth = g["distinct"], g["generated"], g["depth"]
        self.levels, self.deadlocks, self.queue = g["levels"], g["deadlocks"], 0
        self.complete, self.violation, self.trace = True, None, []
        self.stats = {"gpu_ms_total": 1.0, "gpu_ms_expand": 0.5, "gpu_ms_insert": 0.4, "gpu_ms_invariant": 0.1,
                      "launches_expand": g["depth"], "launches_insert": g["depth"] + 1, "launches_other": g["depth"] + 1,
                      "table_slots": 1 << 24, "slot_bytes": 16, "probes": g["generated"] + 7, "max_states": 1 << 23}


def test_single_gpu_line_has_the_contract_keys(monkeypatch, capsys, goldens):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from kafka_specification_b200 import runtime
    g = goldens["kip320_small"]

    class FakeChecker:
        def __init__(self, model, **opts):
            self.words = 2
            self.info = types.SimpleNamespace(exact=1, num_init=1)

        def run(self):
            return _FakeResult(g, self.words)

        def close(self):
            pass

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "Checker", FakeChecker)
    monkeypatch.setattr(bench, "cold_start", lambda model, opts: {"seconds": 1.0, "stub": True})
    args = types.SimpleNamespace(model="kip320_small", warmup=1, steps=2, table_log2=24, max_states=1 << 23,
                                 no_cpu_baseline=False, no_cold=False, dump_outputs=None)
    assert bench.run_single(args) == 0
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in line, k
    assert line["metric"] == "distinct states/sec" and line["n_gpus"] == 1 and line["vs_baseline"] is None
    assert line["config"]["exact_fingerprints"] is True and line["config"]["state_words"] == 2
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert {"kernel", "traffic", "avg_launch_ms", "launches"} <= set(r)
    assert len(line["roofline_other"]) == 2
    c = line["cpu_baseline"]                      # the real CPU arm ran (baseline/cpu_bfs.cpp over the lowered model)
    assert c["kind"] == "port" and c["same_config"] is True and c["value"] > 1e5 and c["cores"] >= 1
    e = line["e2e"]
    assert e["unit"] == "states/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert line["gpu_launches"] == 2 * (3 * g["depth"] + 2)


def test_auxiliary_leg_failure_does_not_cost_the_line(monkeypatch, capsys, goldens):
    import torch
    import bench
    from kafka_specification_b200 import runtime
    g = goldens["kip320_small"]

    class FakeChecker:
        def __init__(self, model, **opts):
            self.words = 2
            self.info = types.SimpleNamespace(exact=1, num_init=1)

        def run(self):
            return _FakeResult(g, self.words)

        def close(self):
            pass

    def boom(*a, **k):
        raise RuntimeError("nvcc exploded")

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "Checker", FakeChecker)
    monkeypatch.setattr(bench, "cold_start", boom)
    monkeypatch.setattr(bench, "cpu_run", boom)
    args = types.SimpleNamespace(model="kip320_small", warmup=1, steps=1, table_log2=24, max_states=1 << 23,
                                 no_cpu_baseline=False, no_cold=False, dump_outputs=None)
    assert bench.run_single(args) == 0
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    assert line["value"] > 0 and "nvcc exploded" in line["e2e_cold"]["error"]
    assert line["cpu_baseline"]["value"] is None and "failed" in line["cpu_baseline"]["sample"]


def test_dump_outputs_is_the_last_step_and_independent_of_store_order(monkeypatch, capsys, goldens, tmp_path):
    """--dump-outputs writes float64 counts, level widths and a state sample chosen by content: two state stores
    holding the same set in different orders give identical files, and every sampled row is an exact stored state."""
    import numpy as np
    import torch
    import bench
    from kafka_specification_b200 import runtime
    g = goldens["kip320_small"]
    store = np.random.default_rng(3).integers(0, np.iinfo(np.uint64).max, size=(g["distinct"], 2),
                                              dtype=np.uint64, endpoint=True)
    runs = []

    class FakeChecker:
        def __init__(self, model, **opts):
            self.words = 2
            self.info = types.SimpleNamespace(exact=1, num_init=1)
            self.store = store[np.random.default_rng(len(runs)).permutation(len(store))]
            self.steps = 0

        def run(self):
            self.steps += 1
            r = _FakeResult(g, self.words)
            r.queue = self.steps                  # tells the steps apart: the dump must be the last one's
            return r

        def copy_states(self, first, count):
            return self.store[first:first + count].copy()

        def close(self):
            pass

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "Checker", FakeChecker)
    for i in range(2):
        out = tmp_path / str(i)
        args = types.SimpleNamespace(model="kip320_small", warmup=1, steps=3, table_log2=24, max_states=1 << 23,
                                     no_cpu_baseline=True, no_cold=True, dump_outputs=str(out))
        assert bench.run_single(args) == 0
        runs.append({f: np.load(out / f) for f in ("counts.npy", "levels.npy", "states_sample.npy")})
    a, b = runs
    assert all(v.dtype == np.float64 for v in a.values())
    # queue = 4: the 4th call of run() (1 warm-up + 3 timed steps)
    assert a["counts.npy"].tolist() == [g["distinct"], g["generated"], g["depth"], 4, g["deadlocks"], 1]
    assert a["levels.npy"].tolist() == g["levels"]
    s = a["states_sample.npy"]
    assert s.shape[1] == 4 and 1 << 16 < len(s) < 1 << 20 and sum(v.nbytes for v in a.values()) < 64 << 20
    assert all(np.array_equal(a[k], b[k]) for k in a)
    words = s.astype(np.uint64).reshape(len(s), 2, 2)
    rows = (words[:, :, 0] << np.uint64(32)) | words[:, :, 1]
    assert set(map(tuple, rows.tolist())) <= set(map(tuple, store.tolist()))


def _run_sharded_worker(model, inject, port):
    import subprocess
    env = dict(os.environ, INJECT="1" if inject else "0")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(ROOT, "tests", "support", "bench_sharded_worker.py"), model],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert out.returncode == 0 and lines, out.stdout[-1500:] + out.stderr[-3000:]
    return json.loads(lines[-1]), out.stderr


@pytest.mark.parametrize("inject", [False, True])
def test_sharded_line_and_collective_fallback(inject, goldens):
    """bench.py --gpus 2 under gloo over the host stand-in: one JSON line from rank 0 with the contract keys; with an
    injected failure of the device-synchronised path in the acceptance (first warm-up) run, every rank falls back to
    the barrier path together and the line says so."""
    g = goldens["kip320_n2"]
    line, err = _run_sharded_worker("kip320_n2", inject, 29671 + int(inject))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "config", "roofline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["n_gpus"] == 2 and line["steps"] == 2 and line["scaling"] == "strong"
    c = line["config"]
    assert c["distinct"] == g["distinct"] and c["generated"] == g["generated"] and sum(c["per_rank_distinct"]) == g["distinct"]
    assert c["nvlink_bytes_per_step_est"] > 0
    if inject:
        assert "device-side sync failed" in c["round_sync_note"] and "injected" in c["round_sync_note"]
        assert c["round_sync"].startswith("stream-ordered NCCL barrier")
        assert "[bench] device-side sync failed" in err
    else:
        assert c["round_sync_note"] is None
