"""bench.py's result line and --dump-outputs.  CPU suite: the reference arm needs no GPU — it must run here, print ONE
JSON line with the benchmark's keys and dump the oracle's outputs.  GPU suite: the timed path dumps its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def _check_dump(d, pkg, oracle):
    """The dump holds, as float64, the OutRecs and the live inventory of bench's N = 1 workload, as the oracle computes them."""
    w = pkg.synth.cfg2()
    out, inv = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    want = {**{f"out_{f}": out[f] for f in out.dtype.names}, **{f"inventory_{f}": inv[f] for f in inv.dtype.names}}
    assert sorted(os.listdir(d)) == sorted(f"{k}.npy" for k in want)
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64 << 20
    for k, v in want.items():
        a = np.load(os.path.join(d, f"{k}.npy"))
        assert a.dtype == np.float64 and np.array_equal(a, v.astype(np.float64)), k


def test_reference_arm_prints_the_contract_line(pkg, oracle, tmp_path):
    d = _bench("--impl", "reference", "--steps", "3", "--warmup", "1", "--dump-outputs", str(tmp_path / "dump"))
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "allocations/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 1
    assert d["value"] > 1e5 and abs(d["ms_per_step"] - 1e3 * 10_000 / d["value"]) < 1e-6 * d["ms_per_step"] + 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert str(cb["cores"]) in cb["by_threads"] and max(cb["by_threads"].values()) == d["value"]
    assert (cb["timed_steps"], cb["warmup"]) == (3, 1) and (cb["port_tuned"]["timed_steps"], cb["port_tuned"]["warmup"]) == (3, 1)
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["claims"] == 10_000 and d["config"]["gpus"] == 1000 and "workload" in d["config"]
    _check_dump(tmp_path / "dump", pkg, oracle)


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=60, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr


class _Counting:
    """Forwards to a ctypes library and counts the calls of one of its functions."""

    def __init__(self, lib, name):
        self.lib, self.name, self.calls = lib, name, 0

    def __getattr__(self, attr):
        f = getattr(self.lib, attr)
        if attr != self.name:
            return f

        def counted(*a):
            self.calls += 1
            return f(*a)
        return counted


def test_cpu_ports_time_exactly_steps_batches(pkg, oracle, monkeypatch):
    """Each thread count of the CPU arm runs `warmup` untimed and `steps` timed batches, no more; the plain port's
    outputs are those of its last timed batch."""
    import bench
    from oracle import tuned
    w = pkg.synth.cfg2(400, 10, 8)
    steps, warmup, cores = 4, 2, 2
    ref, ref_inv = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    plain = _Counting(oracle.lib(), "dra_oracle_allocate_mt")
    monkeypatch.setattr(oracle, "lib", lambda: plain)
    _, _, reps, _, per, out, inv = bench.best_cpu_rate([w], cores, w.n_node, steps, warmup)
    assert reps == steps and len(per) == 2 and plain.calls == len(per) * (warmup + steps)
    assert out.tobytes() == ref.tobytes() and inv.tobytes() == ref_inv.tobytes()
    fast = _Counting(tuned.lib(), "dra_oracle_tuned_allocate")
    monkeypatch.setattr(tuned, "lib", lambda: fast)
    _, _, tper = tuned.best_rate(w, cores, steps, warmup)
    assert len(tper) == 2 and fast.calls == len(tper) * (warmup + steps)


@pytest.mark.gpu
def test_timed_path_dumps_its_last_step(pkg, oracle, tmp_path):
    d = _bench("--steps", "5", "--warmup", "1", "--no-extras", "--dump-outputs", str(tmp_path / "dump"))
    assert d["steps"] == 5 and d["n_gpus"] == 1
    _check_dump(tmp_path / "dump", pkg, oracle)
