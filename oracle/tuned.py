"""ctypes wrapper of oracle/_build/libdra_oracle_tuned.so — the CPU port of spec/ALLOCATION.md written for speed.

TEST INFRASTRUCTURE ONLY (bench.py's cpu_baseline leg and tests/test_oracle_tuned.py).  The plain oracle stays the
parity checker; this one is checked against it and exists so that the reported CPU baseline is not a strawman."""
from __future__ import annotations

import ctypes as C
import os
import statistics
import subprocess
import time

import numpy as np

from . import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libdra_oracle_tuned.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = [os.path.join(_HERE, f) for f in ("dra_oracle_tuned.c", "dra_oracle.c", "dra_oracle.h")]
        if not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in src):
            subprocess.run(["make", "-C", _HERE, "-s"], check=True, stdout=subprocess.DEVNULL)
        _lib = C.CDLL(_SO)
        vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
        _lib.dra_oracle_tuned_allocate.argtypes = [vp, u32, vp, u32, vp, vp, u32, vp, vp, u32, i32]
        _lib.dra_oracle_tuned_allocate.restype = i32
    return _lib


def allocate(gpus, node_off, table, claims, out_off=None, n_out=None, threads: int = 1):
    g = np.ascontiguousarray(gpus, dtype=O.GPU_DTYPE).copy()
    off = np.ascontiguousarray(node_off, dtype=np.uint32)
    t = np.ascontiguousarray(table)
    c = np.ascontiguousarray(claims, dtype=O.CLAIM_DTYPE)
    oo = None if out_off is None else np.ascontiguousarray(out_off, dtype=np.uint32)
    if n_out is None:
        n_out = len(c) if oo is None else 0
    out = np.zeros(max(n_out, 1), dtype=O.OUT_DTYPE)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib().dra_oracle_tuned_allocate(p(g), len(g), p(off), len(off) - 1, p(t), p(c), len(c), p(oo), p(out), n_out, threads)
    if rc != 0:
        raise ValueError(f"dra_oracle_tuned_allocate: rc={rc}")
    return out[:n_out], g


def rate(w, threads: int, steps: int, warmup: int):
    """allocations/s (median over `steps` full batches after `warmup` untimed ones, fresh inventory per batch, like the
    GPU's timed step)."""
    L = lib()
    gpus, claims = w.gpus.copy(), np.ascontiguousarray(w.claims)
    scratch = gpus.copy()
    out = np.zeros(max(w.n_out, 1), dtype=O.OUT_DTYPE)
    off, t = np.ascontiguousarray(w.node_off, dtype=np.uint32), np.ascontiguousarray(w.table)
    oo = None if w.out_off is None else np.ascontiguousarray(w.out_off, dtype=np.uint32)
    p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    ts = []
    for i in range(warmup + steps):
        scratch[:] = gpus
        t0 = time.perf_counter()
        rc = L.dra_oracle_tuned_allocate(p(scratch), len(scratch), p(off), len(off) - 1, p(t), p(claims), len(claims), p(oo), p(out), w.n_out, threads)
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
        assert rc == 0
    return len(claims) / statistics.median(ts), out[: w.n_out].copy(), scratch.copy()


def best_rate(w, cores: int, steps: int, warmup: int):
    """(best rate, its thread count, {threads: rate}); the result is compared with the plain oracle first."""
    ref, ref_inv = O.allocate(w.gpus, w.node_off, w.table, w.claims, w.out_off, w.n_out)
    per, best = {}, None
    top = max(1, min(cores, w.n_node))
    for th in sorted({1, top} | {x for x in (4, 8, 16, 32, 64) if x < top}):
        r, out, inv = rate(w, th, steps, warmup)
        if out.tobytes() != ref.tobytes() or inv.tobytes() != ref_inv.tobytes():
            raise RuntimeError("tuned CPU port differs from the oracle")
        per[th] = r
        if best is None or r > best[0]:
            best = (r, th)
    lib().dra_oracle_tuned_allocate                      # (keep the pool; it is torn down at exit)
    return best[0], best[1], per
