"""CPU suite, part 1: pin the oracle (and the host-side sharing arithmetic) on everything the reference
fixes — its own test vectors, the in-tree geometry fixture — and on the frozen golden files."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES, load_golden


# ---- the reference's own golden vectors: api/nvidia.com/resource/gpu/v1alpha1/sharing_test.go:37-149 ----
def _mps_cases():
    return json.load(open(os.path.join(GOLDEN, "mps_limits.json")))["cases"]


@pytest.mark.parametrize("case", _mps_cases(), ids=lambda c: c["description"])
def test_mps_limit_normalize_matches_reference_vectors(pkg, case):
    sh = pkg.sharing
    errs = {"ErrInvalidDeviceSelector": sh.ErrInvalidDeviceSelector, "ErrInvalidLimit": sh.ErrInvalidLimit}
    if case["expectedError"]:
        with pytest.raises(errs[case["expectedError"]]):
            sh.normalize(case["perDeviceMemoryLimit"], case["uuids"], case["memoryLimit"])
    else:
        got = sh.normalize(case["perDeviceMemoryLimit"], case["uuids"], case["memoryLimit"])
        assert got == case["expectedLimits"]


def test_oracle_megabyte_agrees_with_reference_vectors(pkg, oracle):
    # the arithmetic core of the same vectors, through the C oracle: limit.Megabyte, sharing.go:234-237
    for q, want in [("2Gi", 2048), ("1Gi", 1024), ("10Mi", 10), ("10M", 9), ("1G", 953)]:
        v, ok = oracle.megabyte(pkg.sharing.quantity_value(q))
        assert (v, ok) == (want, True)
        assert pkg.sharing.megabyte_mib(q) == want
    v, ok = oracle.megabyte(pkg.sharing.quantity_value("1M"))
    assert (v, ok) == (0, False)
    with pytest.raises(pkg.sharing.ErrInvalidLimit):
        pkg.sharing.megabyte_mib("1M")


def test_quantity_value_rounds_up_like_apimachinery(pkg):
    q = pkg.sharing.quantity_value
    assert q("1") == 1 and q("1k") == 1000 and q("1Ki") == 1024 and q("1.5Gi") == 1610612736
    assert q("100m") == 1 and q("1e3") == 1000 and q("0.5") == 1 and q("-1500m") == -2
    with pytest.raises(ValueError):
        q("1GiB")


def test_time_slice_interval_int(pkg):
    # TimeSliceInterval.Int, sharing.go:168-180
    assert [pkg.sharing.time_slice_int(s) for s in ("Default", "Short", "Medium", "Long", "x")] == [0, 1, 2, 3, -1]


# ---- the in-tree geometry fixture: gpu-test4.yaml:19-44 + mig-parted-config.yaml:8-16 ----
def test_gpu_test4_geometry(oracle):
    g = load_golden("gpu_test4")
    out, after = oracle.allocate(g["gpus"], g["node_off"], g["table"], g["claims"])
    # every replica lands on its own MIG-enabled GPU as 1g@0, 1g@1, 2g@2, 3g@4 (memory slices 0,1,2-3,4-7)
    for rep in range(4):
        o = out[4 * rep: 4 * rep + 4]
        assert list(o["gpu"]) == [rep] * 4
        assert list(o["start"]) == [0, 1, 2, 4] and list(o["size"]) == [1, 1, 2, 4]
        assert np.all(o["status"] == 0)
    assert list(after["busy"][:4]) == [0xFF] * 4 and list(after["busy"][4:]) == [0] * 4
    # a fifth replica has nowhere to go: MIG devices exist only under MIG-enabled parents (nvlib.go:316-318)
    c5 = np.concatenate([g["claims"], g["claims"][:4]])
    c5["group"][16:] = 99
    out5, _ = oracle.allocate(g["gpus"], g["node_off"], g["table"], c5)
    assert np.all(out5["status"][16:] == 3) and np.all(out5["gpu"][16:] == 0xFFFFFFFF)


def test_cfg1_full_gpu_claims(pkg, oracle):
    w = pkg.synth.cfg1()
    out, after = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    assert list(out["gpu"][:8]) == list(range(8)) and np.all(out["status"][:8] == 0)
    assert np.all(out["status"][8:] == 1) and np.all(out["gpu"][8:] == 0xFFFFFFFF)
    assert np.all(after["flags"] & 2)


def test_full_gpu_excluded_on_mig_enabled(pkg, oracle):
    # nvlib.go:152: a full GPU is published only when MIG is disabled on it
    R = pkg.records
    g, off = R.make_inventory([4], mig=True)
    g["flags"][2] = 0
    c = np.zeros(2, dtype=R.CLAIM_DTYPE)
    c["kind"] = R.KIND_GPU; c["count"] = 1
    out, _ = oracle.allocate(g, off, R.default_table(), c)
    assert list(out["gpu"]) == [2, 0xFFFFFFFF] and list(out["status"]) == [0, 1]


def test_overlap_is_by_memory_slice(pkg, oracle):
    # deviceinfo.go:199-204 / nvml.h:10079-10082: 3g occupies 4 memory slices; slice 7 only via 3g@4 / 7g@0
    R = pkg.records
    g, off = R.make_inventory([1], mig=True)
    c = np.zeros(4, dtype=R.CLAIM_DTYPE)
    c["kind"] = R.KIND_MIG; c["count"] = 1
    c["profile"] = [R.GI_3_SLICE, R.GI_3_SLICE, R.GI_1_SLICE, R.GI_7_SLICE]
    out, after = oracle.allocate(g, off, R.default_table(), c)
    assert [(o["start"], o["size"], o["status"]) for o in out] == [(0, 4, 0), (4, 4, 0), (0, 0, 1), (0, 0, 1)]
    assert after["busy"][0] == 0xFF


# ---- oracle vs the independent pure-Python restatement ----
def _dicts(a):
    return [{k: int(x[k]) for k in a.dtype.names} for x in a]


@pytest.mark.parametrize("seed", range(8))
def test_oracle_matches_naive_restatement(pkg, oracle, seed):
    from oracle import naive
    w = pkg.synth.mixed(500, 9, seed)
    out, after = oracle.allocate(w.gpus, w.node_off, w.table, w.claims, w.out_off, w.n_out)
    tbl = [[(int(w.table[m, p]["size"]), int(w.table[m, p]["start_mask"])) for p in range(16)] for m in range(16)]
    nout, nafter = naive.allocate(_dicts(w.gpus), [int(x) for x in w.node_off], tbl, _dicts(w.claims),
                                  [int(x) for x in w.out_off])
    assert [tuple(int(v) for v in r) for r in out] == nout
    for a, b in zip(after, nafter):
        assert (int(a["busy"]), int(a["flags"]), int(a["mem_free_mib"]), int(a["share_cnt"])) == \
               (b["busy"], b["flags"], b["mem_free_mib"], b["share_cnt"])


@pytest.mark.parametrize("seed,model,wide16,max_width", [(0, 0, False, 8), (3, 0, True, 8), (4, 0, True, 32),
                                                        (2, 1, False, 8), (7, 0, False, 9)])
def test_oracle_matches_naive_on_homogeneous_nodes(pkg, oracle, seed, model, wide16, max_width):
    """The workload class of the CUDA packers' fast loops, incl. a 16-slice part."""
    from oracle import naive
    w = pkg.synth.homog(900, 6, seed, model=model, wide16=wide16, max_width=max_width)
    out, after = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    tbl = [[(int(w.table[m, p]["size"]), int(w.table[m, p]["start_mask"])) for p in range(16)] for m in range(16)]
    nout, nafter = naive.allocate(_dicts(w.gpus), [int(x) for x in w.node_off], tbl, _dicts(w.claims))
    assert [tuple(int(v) for v in r) for r in out] == nout
    assert [int(a["busy"]) for a in after] == [b["busy"] for b in nafter]
    assert (out["status"] == 0).any() and (out["status"] != 0).any()


def test_oracle_mt_equals_single_thread(pkg, oracle):
    w = pkg.synth.cfg2(5000, 60)
    a, ga = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    for threads in (5, 2, 8, 3):              # each change of thread count restarts the worker pool after earlier batches
        b, gb = oracle.allocate(w.gpus, w.node_off, w.table, w.claims, threads=threads)
        assert a.tobytes() == b.tobytes() and ga.tobytes() == gb.tobytes(), threads


# ---- frozen golden files (drift check) ----
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_reproduces_golden(oracle, name):
    g = load_golden(name)
    out, after = oracle.allocate(g["gpus"], g["node_off"], g["table"], g["claims"], g["out_off"], len(g["out"]))
    assert out.tobytes() == g["out"].tobytes()
    assert after.tobytes() == g["gpus_after"].tobytes()


# ---- properties the domain offers ----
def test_deallocate_round_trip(pkg, oracle):
    w = pkg.synth.mixed(1500, 17, 3, invalid=False)
    out, after = oracle.allocate(w.gpus, w.node_off, w.table, w.claims, w.out_off, w.n_out)
    back = oracle.deallocate(after, w.claims, out, w.out_off, n_node=w.n_node)
    assert back.tobytes() == w.gpus.tobytes()


def test_deallocate_counts_slots_like_allocate(pkg, oracle):
    """Found by the property test: a multi-count GPU claim that names no node is INVALID and has ONE OutRec slot
    (spec §1/§3); Deallocate must count its slots the same way (spec §9) — it used to assume `count` slots and ran
    off the end of the result array (or looked at the next claim's record)."""
    R = pkg.records
    g, off = R.make_inventory([2], mig=False)
    c = np.zeros(2, dtype=R.CLAIM_DTYPE)
    c["kind"] = R.KIND_GPU
    c["count"] = [1, 2]
    c["node"] = [0, 1]                                    # the second claim names no node of the inventory
    out_off, n_out = R.out_offsets(c, 1)
    assert (list(out_off), n_out) == ([0, 1], 2)
    out, after = oracle.allocate(g, off, R.default_table(), c, out_off, n_out)
    assert [int(s) for s in out["status"]] == [R.ST_OK, R.ST_INVALID]
    back = oracle.deallocate(after, c, out, out_off, n_node=1)
    assert back.tobytes() == g.tobytes()


def test_idempotent_when_full(pkg, oracle):
    # a second identical batch against the filled inventory allocates nothing new for MIG 7g, and the
    # inventory only ever gains occupancy (monotone)
    w = pkg.synth.cfg2(3000, 20)
    out1, g1 = oracle.allocate(w.gpus, w.node_off, w.table, w.claims)
    out2, g2 = oracle.allocate(g1, w.node_off, w.table, w.claims)
    assert np.all((g1["busy"] & w.gpus["busy"]) == w.gpus["busy"])
    assert np.all((g2["busy"] & g1["busy"]) == g1["busy"])
    assert int((out2["status"] == 0).sum()) <= int((out1["status"] == 1).sum())


def test_unsuitable_nodes_oracle(pkg, oracle):
    R = pkg.records
    g, off = R.make_inventory([2, 2, 0], mig=True)
    g["busy"][0] = 0xFF; g["busy"][1] = 0x0F           # node 0: 4 slices left on gpu 1; node 1 empty
    c = np.zeros(3, dtype=R.CLAIM_DTYPE)
    c["kind"] = R.KIND_MIG; c["count"] = 1
    c["profile"] = [R.GI_3_SLICE, R.GI_3_SLICE, R.GI_7_SLICE]
    pod_off = np.array([0, 2, 3], np.uint32)            # pod0: two 3g; pod1: one 7g
    cand_nodes = np.array([0, 1, 2, 0, 1, 7], np.uint32)
    cand_off = np.array([0, 3, 6], np.uint32)
    bits = oracle.unsuitable(g, off, R.default_table(), c, pod_off, cand_nodes, cand_off)
    got = [(bits[k >> 3] >> (k & 7)) & 1 for k in range(6)]
    assert got == [0, 1, 0, 0, 1, 0]


def test_imex_offset_search(oracle):
    # imexDomainOffsets.add, cmd/nvidia-dra-controller/imex.go:336-349 (128-channel windows below 2048)
    assert oracle.imex_offset([]) == 0
    assert oracle.imex_offset([0, 128, 384]) == 256
    assert oracle.imex_offset(list(range(0, 2048, 128))) == -1


# ---- selectors (spec §10): the legacy GpuClaimParameters.selector shapes, demo/specs/selectors/parameters.yaml:7-27
def test_selectors_inference_and_training_shapes(pkg, oracle):
    R = pkg.records
    g, off = R.make_inventory([4], mig=False)
    attrs = np.zeros(4, dtype=R.ATTR_DTYPE)
    attrs["mem_total_mib"] = [81920, 15258, 40960, 15258]          # "16G" = 15258 MiB by limit.Megabyte arithmetic
    attrs["cc"] = [0x0900, 0x0700, 0x0800, 0x0705]
    attrs["index"] = np.arange(4)
    mem16g = pkg.sharing.megabyte_mib("16G")
    sels = np.stack([
        R.selector(("cmp", R.ATTR_MEMORY_MIB, R.CMP_LE, mem16g), ("cmp", R.ATTR_CC, R.CMP_GE, 0x0705), "and"),  # inference-gpu
        R.selector(("cmp", R.ATTR_MEMORY_MIB, R.CMP_GE, mem16g)),                                                # training-gpu
    ])
    c = np.zeros(4, dtype=R.CLAIM_DTYPE)
    c["kind"] = R.KIND_GPU; c["count"] = 1
    c["mem_limit_mib"] = [1, 2, 1, 9]                    # inference, training, inference again, unknown selector
    oracle.set_selectors(attrs, sels)
    try:
        out, _ = oracle.allocate(g, off, R.default_table(), c)
    finally:
        oracle.set_selectors()
    # inference: <=16G and cc>=7.5 -> only gpu 3; training: >=16G -> lowest is gpu 0; second inference: none left
    assert list(out["gpu"]) == [3, 0, 0xFFFFFFFF, 0xFFFFFFFF]
    assert list(out["status"]) == [0, 0, 1, 5]


def test_selector_programs_edge_cases(pkg, oracle):
    R = pkg.records
    w = pkg.synth.mixed(400, 6, 2, invalid=False)
    attrs, sels = pkg.synth.with_selectors(w, 3)
    oracle.set_selectors(attrs, sels)
    try:
        out, inv = oracle.allocate(w.gpus, w.node_off, w.table, w.claims, w.out_off, w.n_out)
    finally:
        oracle.set_selectors()
    sid = np.where(w.claims["kind"] == R.KIND_SHARED, w.claims["group"], w.claims["mem_limit_mib"])
    first = out[w.out_off]
    assert np.all(first["status"][sid > len(sels)] == 5)                  # ids beyond the table: INVALID
    assert not np.any(first["status"][sid == 5] == 0)                      # the malformed program passes nothing
    assert np.any(first["status"][(sid > 0) & (sid <= len(sels))] == 0)    # and real selectors do allocate
