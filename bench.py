#!/usr/bin/env python
"""bench.py — claim allocations/sec on the BASELINE.json workload.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one Allocate batch: 10,000 mixed 1g/2g/3g/7g MIG claims (generation order, NOT node-sorted)
over 125 nodes x 8 GPUs, evaluated against the freshly loaded inventory (BASELINE.md cfg2 = configs[1]).
At N GPUs the step is ONE GLOBAL batch of N x 10k claims over N x 125 nodes (weak scaling; at N = 8 this is
BASELINE configs[2]'s shape): every rank holds the whole inventory and receives the SAME claim array, filters the
claims of its own node range on the device, allocates them and writes every OutRec at the claim's global slot of
every rank's table — the path's one collective, an all-gather of 16-byte packets over NVLink inside the
allocation kernel (dra_allocate_batch_global_device).  No host-side partition or merge is involved.

value   = whole-job allocations/s with inputs resident in HBM (CUDA events on the launch stream, L2
          flushed between steps, max over ranks)
e2e     = the same through the C-ABI host call dra_allocate_batch with pinned host buffers, every step moving the
          160 KB of claims host -> device and the 80 KB of OutRecs device -> host inside the timed region: by the
          kernel itself (direct host I/O: one cooperative launch reads / writes the pinned buffers), or with
          --no-direct by copy-engine transfers around it (H2D -> kernels -> D2H as one CUDA graph)
roofline= algorithmic bytes of the batch / device time of the dominant kernel, vs MEASURED_PEAKS.json
cpu_baseline / --impl reference = the CPU oracle of the same spec on the host cores (kind "port": the
          reference's Go allocator does not exist in the snapshot, SURVEY.md F1; no Go toolchain)
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "claim allocations/sec — 10k mixed GPU+MIG claims over 1k-GPU inventory"
UNIT = "allocations/s"
CLAIMS_PER_RANK, NODES_PER_RANK, GPUS_PER_NODE = 10_000, 125, 8


def workload(pkg, world: int):
    """The GLOBAL batch of the job: world x (10k claims, 125 nodes x 8 GPUs); world 1 = cfg2 exactly."""
    w = pkg.synth.cfg2(CLAIMS_PER_RANK * world, NODES_PER_RANK * world, GPUS_PER_NODE)
    if world > 1:
        w.name = f"cfg2 x{world} (one global batch)"
    return w


def config(world: int, aligned: bool = False) -> dict:
    return {"workload": "cfg2: 10k mixed 1g/2g/3g/7g MIG claims (40/30/20/10 %), unsorted, 125 nodes x 8 GPUs"
                        + (f"; x{world}: ONE global batch of {CLAIMS_PER_RANK * world} claims over {NODES_PER_RANK * world} nodes, node ranges "
                           f"sharded over {world} ranks on the device + all-gather of OutRecs" if world > 1 else ""),
            "claims": CLAIMS_PER_RANK * world, "gpus": NODES_PER_RANK * GPUS_PER_NODE * world,
            "nodes": NODES_PER_RANK * world, "parallelism": f"node-shard x{world}",
            "l2": "flushed between steps (256 MiB write)" + ("; ranks lined up on the device after each flush (untimed dra_peer_rendezvous_device), so a "
                                                             "step does not time its peers' flush skew" if world > 1 and aligned else ""),
            "inventory": "fresh per step (DRA_F_FRESH_INVENTORY)"}


def dump_outputs(d: str, out: np.ndarray, inv: np.ndarray | None = None) -> None:
    """What a caller of the timed call receives, one float64 array per record field (every field is an integer of at
    most 32 bits, so the values are exact): out_<field>.npy for the OutRecs, inventory_<field>.npy for the live
    inventory the call leaves behind (N = 1 only; at N > 1 a rank's inventory is authoritative for its own nodes)."""
    os.makedirs(d, exist_ok=True)
    for prefix, rec in (("out", out), ("inventory", inv)):
        if rec is not None:
            for f in rec.dtype.names:
                np.save(os.path.join(d, f"{prefix}_{f}.npy"), rec[f].astype(np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self) -> dict:
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].startswith("Active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_oracle_rate(w_list, threads: int, steps: int, warmup: int):
    """allocations/s of the CPU oracle on the concatenated workload: `warmup` untimed batches, then `steps` timed ones;
    returns (rate, steps, seconds, OutRecs, inventory) with the outputs of the last timed batch."""
    from oracle import oracle as O
    O.build()
    pkg = importlib.import_module("k8s-dra-driver_b200")
    R = pkg.records
    gpus = np.concatenate([w.gpus for w in w_list]).copy()
    claims = np.concatenate([w.claims for w in w_list]).copy()
    node_off = [np.zeros(1, np.uint32)]
    nb, gb = 0, 0
    off_c = 0
    for w in w_list:
        node_off.append(w.node_off[1:] + np.uint32(gb))
        gpus["node"][gb: gb + w.n_gpu] += np.uint32(nb)
        claims["node"][off_c: off_c + w.n_claim] += np.uint32(nb)
        nb += w.n_node; gb += w.n_gpu; off_c += w.n_claim
    node_off = np.concatenate(node_off).astype(np.uint32)
    table = np.ascontiguousarray(w_list[0].table)
    lib = O.lib()
    out = np.zeros(len(claims), dtype=R.OUT_DTYPE)
    scratch = gpus.copy()
    p = lambda a: a.ctypes.data  # noqa: E731
    times = []
    for i in range(warmup + steps):
        scratch[:] = gpus                                   # fresh inventory per step, as on the GPU
        t0 = time.perf_counter()
        rc = lib.dra_oracle_allocate_mt(p(scratch), len(scratch), p(node_off), len(node_off) - 1, p(table),
                                        p(claims), len(claims), None, p(out), len(out), threads)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
        assert rc == 0
    med = statistics.median(times)
    return len(claims) / med, len(times), sum(times), out, scratch


def thread_candidates(cores: int, n_node: int):
    """Thread counts to try for the pooled multi-threaded oracle: nodes are the unit of parallel work."""
    top = max(1, min(cores, n_node))
    return sorted({1, top} | {t for t in (8, 16, 32, 64) if t < top})


def best_cpu_rate(w_list, cores: int, n_node: int, steps: int, warmup: int):
    """(rate, threads, reps, seconds, {threads: rate}, OutRecs, inventory) of the fastest thread count; the outputs are
    those of its last timed batch."""
    per, best = {}, None
    for th in thread_candidates(cores, n_node):
        rate, reps, secs, out, inv = cpu_oracle_rate(w_list, th, steps, warmup)
        per[th] = rate
        if best is None or rate > best[0]:
            best = (rate, th, reps, secs, out, inv)
    return (*best[:4], per, *best[4:])


def cpu_arm(pkg, w, cores: int, steps: int, warmup: int):
    """The CPU arm on one global workload: the oracle port (the checker, plain restatement of the spec) and, beside
    it, the tuned port of the same spec (oracle/dra_oracle_tuned.c: no allocation in the call, parallel bucketing,
    -O3 -march=native, shift/AND fit map) — both with every thread count in by_threads, the best one reported, each
    thread count timed over `steps` batches after `warmup` untimed ones.  Returns (result dict, OutRecs, inventory),
    the outputs of the oracle port's last timed batch at its best thread count."""
    rate, th, reps, secs, per, out, inv = best_cpu_rate([w], cores, w.n_node, steps, warmup)
    d = {"value": rate, "unit": UNIT, "cores": th, "kind": "port", "timed_steps": reps, "warmup": warmup,
         "sample": f"{reps} timed full batches of {w.n_claim} claims after {warmup} untimed, median; CPU oracle of spec/ALLOCATION.md (plain restatement, the "
                   f"parity checker), nodes spread over a persistent thread pool; best of the thread counts in by_threads "
                   f"(the reference's Go allocator is absent from the snapshot and Go is not installed)",
         "value_1_thread": per[1], "by_threads": {str(k): v for k, v in per.items()}, "host_cores": cores}
    try:
        from oracle import tuned as T
        tr, tth, tper = T.best_rate(w, cores, steps, warmup)
        d["port_tuned"] = {"value": tr, "unit": UNIT, "cores": tth, "kind": "port-tuned", "by_threads": {str(k): v for k, v in tper.items()},
                           "timed_steps": steps, "warmup": warmup,
                           "note": "same spec, same bytes out (checked against the oracle before timing); a reported baseline, "
                                   "what a CPU implementation written for speed concedes"}
    except Exception as e:                                  # the tuned port is optional test infrastructure
        d["port_tuned"] = {"unavailable": str(e)[:200]}
    return d, out, inv


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = args.gpus
    if rank != 0:
        return 0
    pkg = importlib.import_module("k8s-dra-driver_b200")
    w = workload(pkg, world)
    cores = os.cpu_count() or 1
    from oracle import oracle as O
    O.build()
    cpu, out, inv = cpu_arm(pkg, w, cores, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, inv if world == 1 else None)
    rate = cpu["value"]
    n = w.n_claim
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n / rate, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": config(world), "cpu_baseline": cpu,
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


class Timer:
    """K steps, each bracketed by CUDA events on the launch stream, L2 flushed before each; max over ranks."""

    def __init__(self, torch, dist, stream, dev, world, flush):
        self.torch, self.dist, self.stream, self.dev, self.world, self.flush = torch, dist, stream, dev, world, flush
        self.align = None        # N > 1: device-side rendezvous of the ranks, enqueued between the flush and the timed step

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, step, steps, warmup):
        torch = self.torch
        for _ in range(max(3, warmup)):
            self.flush.fill_(1); step()
        self.barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for a, b in evs:
            self.flush.fill_(1)                   # L2 flush, outside the event pair
            if self.align:                        # the ranks' 256 MiB flushes do not take the same time: without this a rank's
                self.align()                      # event pair would also time its wait for the peer whose flush ran longest
            a.record(self.stream); step(); b.record(self.stream)
        self.barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()) / steps


def run_ours(args):
    os.environ.setdefault("NCCL_DEBUG", "WARN")     # keep stdout to the one JSON line
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("k8s-dra-driver_b200")
    R = pkg.records
    from oracle import oracle as O
    world = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one explicit stream for everything (flush, events, our kernels): the legacy default stream's handle is
    # 0, which the C ABI reads as "create your own stream", and events on another stream would time nothing
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    timer = Timer(torch, dist, stream, dev, world, flush)
    F = pkg.api.F_FRESH_INVENTORY

    w = workload(pkg, world)
    n_claim, n_out = w.n_claim, w.n_out
    # DRA_CFG_USE_GRAPH only concerns the host-buffer call (the e2e leg): H2D -> kernel -> D2H as one graph launch
    ctx = pkg.api.Context(device=local, stream=stream.cuda_stream, max_claims=n_claim,
                          flags=(0 if args.no_graph else pkg.api.CFG_USE_GRAPH) | (pkg.api.CFG_NO_DIRECT if args.no_direct else 0)
                                | (0 if (args.no_resident or args.no_direct) else pkg.api.CFG_RESIDENT))
    collective = None
    if world > 1:
        uid = [pkg.api.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
        collective = "all-gather of OutRecs as 16-byte self-validating packets over NVLink, inside the allocation kernel (own code)"

    def load(wl):
        """Inventory + (N > 1) this rank's node range and the gather buffers for one global workload."""
        ctx.set_table(wl.table)
        ctx.set_inventory(wl.gpus, wl.node_off)
        if world > 1:
            ranges = pkg.shard.plan(wl.claims["node"], wl.n_node, world)      # one-time set-up, like the inventory
            ctx.set_shard_map([r[0] for r in ranges] + [ranges[-1][1]], stray_rank=0)
            hs = [None] * world
            dist.all_gather_object(hs, ctx.shard_export(wl.n_out))
            ctx.peer_import(hs)
            timer.align = ctx.peer_rendezvous if args.align else None

    def make_step(wl, d_claims, d_out):
        if world > 1:
            return lambda: ctx.allocate_global_device(d_claims.data_ptr(), wl.n_claim, None, wl.n_out, F)
        return lambda: ctx.allocate_device(d_claims.data_ptr(), wl.n_claim, None, d_out.data_ptr(), wl.n_out, F)

    def result(wl, d_out):
        if world > 1:
            return ctx.gather_read(np.zeros(wl.n_out, dtype=R.OUT_DTYPE))
        return d_out.cpu().numpy().view(R.OUT_DTYPE)

    load(w)
    d_claims = torch.from_numpy(w.claims.view(np.uint8).copy()).to(dev)
    d_out = torch.zeros(n_out * 8, dtype=torch.uint8, device=dev)
    step_dev = make_step(w, d_claims, d_out)

    # ---- parity guard: the timed path must produce the oracle's bytes (every rank checks the WHOLE table) ----
    step_dev(); ctx.sync()
    ref_out = O.allocate(w.gpus, w.node_off, w.table, w.claims)[0]
    if result(w, d_out).tobytes() != ref_out.tobytes():
        raise SystemExit("bench: CUDA result differs from the oracle — refusing to time a wrong kernel")

    # ---- device-resident throughput ---------------------------------------------------------------------
    launches0 = ctx.launch_count()
    with ClockSampler(local) as clk:
        ms_per_step = timer.run(step_dev, args.steps, args.warmup)
        if args.steps * ms_per_step < 250:                     # a short run: keep the sampler up long enough for > 1 sample
            time.sleep(0.25)
    ctx.sync()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, result(w, d_out), ctx.get_inventory() if world == 1 else None)
    launches = (ctx.launch_count() - launches0) * args.steps // (args.steps + max(3, args.warmup))
    value = n_claim / (ms_per_step * 1e-3)

    # ---- per-kernel device times (separate pass: event pairs around every kernel) --------------------
    ctx.set_profiling(True)
    stage = {}
    for _ in range(args.steps):
        if world > 1:
            dist.barrier()                         # (the gather waits for its peers: without this a rank's host-side delay would be timed)
        flush.fill_(1); step_dev(); ctx.sync()
        for k, v in ctx.timings_us().items():
            stage.setdefault(k, []).append(v)
    ctx.set_profiling(False)
    if world > 1:
        dist.barrier()
    stage_us = {k: statistics.mean(v) for k, v in stage.items() if statistics.mean(v) > 0}
    per_step = launches // max(1, args.steps)
    if "pack" in stage_us and "bucket_hist" not in stage_us and "bucket_scatter" not in stage_us:   # single-launch path
        stage_us = {"fused": stage_us["pack"]}
    dom = max((k for k in stage_us if k != "all_gather"), key=lambda k: stage_us[k])
    note_evt = "each stage time includes ~2.7 us of CUDA-event pair overhead (profiles/launch_overhead_r01d.txt)"
    peak, peak_src = peaks()
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = {"fused": "k_fused"}.get(dom, dom)
        if key in tj and world == 1:
            traffic = tj[key]["dram__bytes_read.sum"] + tj[key]["dram__bytes_write.sum"]
            traffic_src = tj[key]["source"]
    except Exception:
        pass
    alg_bytes = w.algorithmic_bytes() if world == 1 else (16 * n_claim + 16 * w.n_gpu // world + 8 * n_out // world)
    achieved = alg_bytes / (stage_us[dom] * 1e-6) / 1e9 if stage_us[dom] > 0 else 0.0

    # ---- end to end through the C-ABI host call ---------------------------------------------------------
    pin_c = pkg.api.PinnedBuffer(n_claim, R.CLAIM_DTYPE)
    pin_c.array[:] = w.claims
    pin_o = pkg.api.PinnedBuffer(n_out, R.OUT_DTYPE)
    h_claims_t = torch.from_numpy(pin_c.array.view(np.uint8))

    def step_e2e():
        if world == 1:
            ctx.allocate_raw(pin_c.ptr, n_claim, None, pin_o.ptr, n_out, F)      # the bare C-ABI call
        elif args.e2e_copy:
            d_claims.copy_(h_claims_t, non_blocking=True)
            step_dev()
            ctx.gather_read(pin_o.array)
        else:
            # the sharded call takes the pinned host buffer itself: the compaction kernel reads every claim exactly once, straight
            # over PCIe (no copy-engine transfer in front of it); the table comes back with dra_gather_read
            ctx.allocate_global_device(pin_c.ptr, n_claim, None, n_out, F)
            ctx.gather_read(pin_o.array)

    for _ in range(max(3, args.warmup)):
        step_e2e()
    timer.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    if world == 1:
        ctx.serve_stop()                       # resident mode: the EXIT is part of the timed region (the barrier below needs an idle device)
    timer.barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = n_claim * args.steps / e2e_s
    assert pin_o.array.tobytes() == ref_out.tobytes()

    # ---- the other BASELINE configs and calls, driver-timed with the same discipline (extra keys) -------------
    extras = {}
    if not args.no_extras:
        extras = run_extras(pkg, O, ctx, timer, torch, dev, world, rank, load, make_step, result, args)

    line = None
    if rank == 0:
        cores = os.cpu_count() or 1
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": dict(config(world, args.align), **({"collective": collective} if collective else {})),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 16 * n_claim,
                        "d2h_bytes_per_step": 8 * n_out, "timer": "host wall clock around the C-ABI call",
                        "us_per_batch": 1e6 * e2e_s / args.steps,
                        "cuda_graph": bool(world == 1 and not args.no_graph and args.no_direct),
                        "resident_batches": ctx.serve_batches(),
                        "host_io": ("resident kernel + doorbell: the single-launch kernel stays up, a call writes a 64-byte command and a sequence number into "
                                    "mapped host memory and spins on the completion word; the kernel reads the claims from / writes the OutRecs to the pinned host buffers"
                                    if world == 1 and not args.no_direct and not args.no_resident else
                                    "direct: one cooperative launch, the kernel reads the claims from / writes the OutRecs to the pinned host buffers"
                                    if world == 1 and not args.no_direct else
                                    "copy engine: H2D of the global claim array, kernels, D2H of the whole table" if args.e2e_copy else
                                    "the compaction kernel reads the global claim array from the pinned host buffer itself (zero-copy ingest), kernels, "
                                    "D2H of the whole table (dra_gather_read)")},
                "gpu_launches": launches,
                "clocks": clk.summary(),
                "roofline": {"bound": "hbm", "kernel": {"fused": "k_fused", "pack": "k_pack", "bucket_hist": "k_bucket_hist",
                                                         "bucket_scan": "k_bucket_scan",
                                                         "bucket_scatter": "k_bucket_scatter"}.get(dom, dom),
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                             "note": "24 B/claim + 16 B/GPU = 256 KB per batch is ~40 ns of HBM time: the path is "
                                     "bound by launch latency and the per-node first-fit dependency chain, not by bytes"
                                     + ("; at N > 1 per rank: the global claim array read once + its own GPUs and OutRecs" if world > 1 else "")},
                "stages_us": stage_us, "stages_note": note_evt,
                "us_per_batch": ms_per_step * 1e3}
        line.update(extras)
        if world == 1:
            line["cpu_baseline"] = cpu_arm(pkg, w, cores, args.steps, args.warmup)[0]
        print(json.dumps(line))
    pin_c.free(); pin_o.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_extras(pkg, O, ctx, timer, torch, dev, world, rank, load, make_step, result, args) -> dict:
    """Every other BASELINE config, the sharded configs[2] and a size where sharding should pay, UnsuitableNodes and the
    pod mode — same timing discipline as the headline (events, L2 flush, max over ranks, --steps timed steps), parity against
    the oracle before each timing.  Keys are added to the one JSON line."""
    R, S = pkg.records, pkg.synth
    steps = args.steps
    F = pkg.api.F_FRESH_INVENTORY
    out = {}

    def alloc_case(wl, check=True):
        load(wl)
        d_c = torch.from_numpy(wl.claims.view(np.uint8).copy()).to(dev)
        d_o = torch.zeros(max(1, wl.n_out) * 8, dtype=torch.uint8, device=dev)
        step = make_step(wl, d_c, d_o)
        l0 = ctx.launch_count()
        step(); ctx.sync()
        per = ctx.launch_count() - l0
        ok = None
        if check:
            ok = result(wl, d_o).tobytes() == O.allocate(wl.gpus, wl.node_off, wl.table, wl.claims, threads=8)[0].tobytes()
            if not ok:
                raise SystemExit(f"bench: {wl.name}: CUDA result differs from the oracle")
        ms = timer.run(step, steps, 3)
        ab = wl.algorithmic_bytes()                                     # 16 B/claim + 16 B/GPU + 8 B/slot (SURVEY 8d)
        return {"claims": wl.n_claim, "gpus": wl.n_gpu, "nodes": wl.n_node, "us_per_batch": ms * 1e3,
                "alloc_per_s": wl.n_claim / (ms * 1e-3), "kernel_launches_per_batch": per, "parity": "bit-exact vs oracle",
                "algorithmic_bytes": ab, "hbm_frac_whole_step": ab / (ms * 1e-3) / 1e9 / peaks()[0]}

    cfgs = {}
    if world == 1:
        for name in ("cfg1", "cfg3", "cfg4", "cfg5"):
            cfgs[name] = alloc_case(S.CONFIGS[name]())
    else:
        cfgs["cfg3"] = alloc_case(S.cfg3())
    big = S.cfg2(1_000_000, 10_000, 8, seed_off=9); big.name = "1M claims x 80k GPUs"
    cfgs["large_1M_x_80k"] = alloc_case(big)
    out["configs"] = cfgs
    out["configs_note"] = ("device-resident, one batch per step, fresh inventory, L2 flushed; at N > 1 every config is ONE global batch "
                           "sharded by node range on the device; compare the same key of the N = 1 line for the crossover")
    if world == 1:
        # UnsuitableNodes: 10,000 pods x 125 candidate nodes (dense) against a half-full cfg2 inventory
        w = S.cfg2()
        _, inv = O.allocate(w.gpus, w.node_off, w.table, w.claims[:4000])
        ctx.set_table(w.table); ctx.set_inventory(inv, w.node_off)
        n_pod = 10_000
        claims = w.claims[:n_pod].copy()
        pod_off = np.arange(n_pod + 1, dtype=np.uint32)
        n_pair = n_pod * w.n_node
        uns = {}
        for key, fl, ofl in (("first_fit", 0, 0), ("exhaustive", pkg.api.F_EXHAUSTIVE, O.F_EXHAUSTIVE)):
            bits = ctx.unsuitable(claims, pod_off, flags=fl)
            cn = np.tile(np.arange(w.n_node, dtype=np.uint32), 500); co = (np.arange(501, dtype=np.uint32) * w.n_node).astype(np.uint32)
            ref = O.unsuitable(inv, w.node_off, w.table, claims[:500], pod_off[:501], cn, co, flags=ofl)
            assert bits[: len(ref) - 1].tobytes() == ref[: len(ref) - 1].tobytes()
            ts = []
            for _ in range(args.steps):
                t0 = time.perf_counter(); ctx.unsuitable(claims, pod_off, flags=fl); ts.append(time.perf_counter() - t0)
            ctx.set_profiling(True); ctx.unsuitable(claims, pod_off, flags=fl)
            k_us = list(ctx.timings_us().values())[0]
            ctx.set_profiling(False)
            uns[key] = {"pairs": n_pair, "e2e_ms": statistics.median(ts) * 1e3, "kernel_us": k_us,
                        "kernel_pairs_per_s": n_pair / (k_us * 1e-6), "suitable_pairs": int(np.unpackbits(bits).sum())}
        out["unsuitable"] = uns
        # pod mode (spec §12) on the fragmented inventory: how many (pod, node) verdicts the exhaustive search flips
        pw, ppo = S.pods(20_000, 64, 1)
        sub = 4000
        po = ppo[: sub + 1]; pc = pw.claims[: po[-1]]
        ctx.set_table(pw.table); ctx.set_inventory(pw.gpus, pw.node_off)
        ff = np.unpackbits(ctx.unsuitable(pc, po), bitorder="little")[: sub * 64]
        def med(fn):                                        # (the first call of a shape also grows buffers: median of the later ones)
            r = fn(); ts = []
            for _ in range(args.steps):
                t0 = time.perf_counter(); r = fn(); ts.append(time.perf_counter() - t0)
            return r, statistics.median(ts)
        exb, t_ex = med(lambda: ctx.unsuitable(pc, po, flags=pkg.api.F_EXHAUSTIVE))
        ex = np.unpackbits(exb, bitorder="little")[: sub * 64]
        po_out, t_ap = med(lambda: ctx.allocate_pods(pw.claims, ppo, flags=pkg.api.F_EXHAUSTIVE | F))
        _, t_ap_ff = med(lambda: ctx.allocate_pods(pw.claims, ppo, flags=F))
        ref, _ = O.allocate_pods(pw.gpus, pw.node_off, pw.table, pw.claims, ppo, flags=O.F_EXHAUSTIVE)
        assert po_out.tobytes() == ref.tobytes()
        out["pod_mode"] = {"workload": "pods of 1-5 mixed MIG claims on cfg5's pre-fragmented 512 GPUs (synth.pods)",
                           "pairs": sub * 64, "suitable_first_fit": int(ff.sum()), "suitable_exhaustive": int(ex.sum()),
                           "flipped_to_suitable": int((ex & ~ff).sum()), "unsuitable_exhaustive_e2e_ms": t_ex * 1e3,
                           "allocate_pods_exhaustive_e2e_ms": t_ap * 1e3, "allocate_pods_first_fit_e2e_ms": t_ap_ff * 1e3,
                           "note": f"host wall clock of the C-ABI call, median of {args.steps} after a first call; 64 nodes = 64 sequential chains of ~312 pods: "
                                   "the exhaustive call is bound by the longest chain of searches, not by the GPU's width", "pods": 20_000, "claims": int(pw.n_claim),
                           "search_limit_slots": int((po_out["status"] == R.ST_SEARCH_LIMIT).sum()), "parity": "bit-exact vs oracle"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of every timed loop: the headline, the e2e leg, the per-kernel "
                    "stage pass, the other configs, UnsuitableNodes, pod mode and, per thread count, the CPU ports")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-direct", action="store_true", help="e2e leg: copy-engine transfers around the kernel instead of direct host I/O")
    ap.add_argument("--no-graph", action="store_true", help="e2e leg: enqueue H2D / kernel / D2H separately instead of one CUDA graph")
    ap.add_argument("--no-resident", action="store_true", help="e2e leg: one cooperative launch per batch instead of the resident kernel + doorbell")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload (skip the other configs / calls)")
    ap.add_argument("--e2e-copy", action="store_true", help="N > 1, e2e leg: H2D copy of the global claim array in front of the call instead of zero-copy ingest")
    ap.add_argument("--align", action="store_true", help="N > 1: device-side rendezvous of the ranks (dra_peer_rendezvous_device) between the untimed L2 "
                    "flush and the timed step; measured at N = 2: no difference (29.46 vs 29.48 us), off by default")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(float64; the inputs are seeded, so runs with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
