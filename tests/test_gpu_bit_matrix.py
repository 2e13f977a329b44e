"""The bit-sliced path (csrc/engine.cu: bit_eval_kernel in its single-set, batch-ring and batch-register variants, the
contract check and field-input transpose of its prologue, bit_expand_kernel, bit_expand_wide_kernel, the bad-set list the
generic kernel takes over, the speculation drop and the launch heuristics of Engine::launch_bit) under every bit-plan
option, launch shape and contract pattern, row by row against the C oracle.

The plan compiler is checked on the host simulator (tests/test_bitplan.py); the simulator's step loop reads every lane's
operands before any lane writes and has no rings, warps or expansion kernels of its own.  Here util.bit_corpus runs on the
GPU.  Every witness row must equal the oracle's and every flag word the throughput simulator's; device outputs start as 0xFF
bytes (no canonical value), so a position a kernel skips shows up.  GW_TRACE_HOST=1 makes the engine print one line per bit
launch, so the tests know which variant ran and in what shape."""
import ctypes
import importlib
import json
import os
import random
import re

import numpy as np
import pytest

from oracle import cref
from tests import util
from tests.test_bitplan import boolean_graph
from tests.util import po

pytestmark = pytest.mark.gpu

M = util.M
ENV_KEYS = ("GW_BITSLICE", "GW_BIT_RING", "GW_BIT_WARPS", "GW_BIT_MERGE", "GW_BIT_MIN_SETS", "GW_BIT_MAX_SLOTS", "GW_LAT_BIT",
            "GW_TRACE_HOST", "GW_CHUNK_MB", "GW_SINGLE_MODE", "GW_DEVICE", "GW_THREADS", "GW_REGS")
TRACE = re.compile(r"\[gw bit\] variant (\w+), warps (\d+), ctas (\d+), groups (\d+)")
BATCHES = (1, 2, 31, 32, 33, 65, 1029)
BAD_VALUES = [2, M - 1, M, M + 1, (1 << 256) - 1] + [1 + (1 << (32 * k)) for k in range(1, 8)]
FIELD_VALUES = [0, 1, M - 1, M, M + 1, 1 << 253, (1 << 256) - 1]


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


@pytest.fixture(scope="module")
def dev():
    torch = pytest.importorskip("torch")
    p = torch.cuda.get_device_properties(0)
    return {"sms": p.multi_processor_count, "smem": int(p.shared_memory_per_block_optin)}


def _set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("GW_TRACE_HOST", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))


def _pack(rows):
    return np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32)


def _bit_eligible(cwc, g):
    """gw_graph_info now (Graph.info is read once, when the graph is loaded)"""
    info = cwc.gw_graph_info_t()
    cwc._L.gw_graph_info(g._h, ctypes.byref(info))
    return int(info.bit_eligible)


def _traces(capfd):
    return [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in TRACE.finditer(capfd.readouterr().err)]


def expected_launch(info, B, dev, env):
    """(variant, warps per CTA, CTAs, groups) that Engine::launch_bit picks for a plan with simulator info `info`"""
    smem, sms = dev["smem"], dev["sms"]
    n_groups = (B + 31) // 32
    planes_b = (info["n_slots"] * 4 + 15) & ~15
    single_b, ring_b = planes_b + 32 + 3 * 16 * 512, planes_b + 32 + 3 * 8 * 512
    if B == 1 and single_b <= smem:
        return ("single", 1, 1, 1)
    fit_ring, fit_reg = smem // ring_b, smem // planes_b
    per_sm = -(-n_groups // sms)
    ring = ring_b <= smem and info["n_steps"] >= 128 and (per_sm <= fit_ring or fit_ring * 2 >= fit_reg)
    if env.get("GW_BIT_RING") == "0":
        ring = False
    elif env.get("GW_BIT_RING") == "1" and ring_b <= smem:
        ring = True
    wpb = min(8, smem // (ring_b if ring else planes_b))
    while wpb > 1 and n_groups < wpb * 2 * sms:
        wpb -= 1
    if 1 <= int(env.get("GW_BIT_WARPS", 0)) <= wpb:
        wpb = int(env["GW_BIT_WARPS"])
    return ("ring" if ring else "reg", wpb, -(-n_groups // wpb), n_groups)


class Case:
    """a graph of the corpus, its input rows, the oracle's witness rows, the throughput simulator's flag words, and the bit
    plan's simulator info (merged and unmerged)"""

    def __init__(self, name, data, rows):
        self.name, self.data = name, data
        self.inp = _pack(rows)
        self.want = cref.CGraph(data).evaluate_batch(self.inp, os.cpu_count() or 4)
        sim = util.SimGraph(data, **util.sim_options({}))
        self.flags = np.array([sim.eval(r)[1] for r in rows], dtype=np.uint32)
        self.bits = {True: util.BitSimGraph(data), False: util.BitSimGraph(data, merge=False)}

    def check(self, out, flags, B, what="", rows=None):
        rows = np.arange(B) if rows is None else np.asarray(rows)
        out = out.reshape(B, -1)[rows]
        bad = np.nonzero((out != self.want[rows].reshape(len(rows), -1)).any(axis=1))[0]
        assert len(bad) == 0, f"{self.name} {what} B={B}: {len(bad)} wrong witness rows, first {rows[bad[:8]].tolist()}"
        if flags is not None:
            f = np.asarray(flags).reshape(-1)[rows]
            badf = np.nonzero(f != self.flags[rows])[0]
            assert len(badf) == 0, f"{self.name} {what} B={B}: wrong flags in rows {rows[badf[:8]].tolist()}"


def contract_inputs(data):
    """(contract inputs, field inputs, inputs per row) of a graph's bit plan"""
    s = util.BitSimGraph(data)
    inp = s.plan()["inputs"]
    con = sorted({int(i) for i in inp[inp[:, 2] == util.BIT_CONTRACT, 0]})
    fld = sorted({int(i) for i in inp[inp[:, 2] != util.BIT_CONTRACT, 0]})
    return con, fld, s.I


def corpus_rows(rnd, data, n, bad_rows):
    """n input rows: bits on the contract inputs, edge and random values on the field inputs, and a value from BAD_VALUES on
    one contract input of each row of bad_rows (cycling through the list)"""
    con, fld, n_in = contract_inputs(data)
    rows = []
    for b in range(n):
        r = [1] + [rnd.randrange(2) for _ in range(n_in - 1)]
        for i in fld:
            r[i] = FIELD_VALUES[(b + i) % len(FIELD_VALUES)] if b % 3 else util.random_value(rnd)
        rows.append(r)
    k = 0
    for b in bad_rows:
        if b < n and con:
            rows[b][con[(b * 7) % len(con)]] = BAD_VALUES[k % len(BAD_VALUES)]
            k += 1
    return rows


# bad sets of the corpus rows: lanes 1 and 31 of group 0, lane 0 of group 1 (the ragged last group of B = 33 and 65), the
# whole group 3 between good groups, and single sets up to the ragged last group of B = 1029
CORPUS_BAD = [1, 31, 32, 64] + list(range(96, 128)) + [200, 517, 1023, 1028]


@pytest.fixture(scope="module")
def corpus():
    rnd = random.Random(9090)
    out = []
    for name, data in util.bit_corpus():
        n = 65 if name.startswith("sha256") else max(BATCHES)
        out.append(Case(name, data, corpus_rows(rnd, data, n, CORPUS_BAD)))
    return out


BIT_VARIANTS = [("defaults", {}), ("ring_1", {"GW_BIT_RING": "1"}), ("ring_0", {"GW_BIT_RING": "0"}), ("merge_0", {"GW_BIT_MERGE": "0"}),
                ("min_sets_33", {"GW_BIT_MIN_SETS": "33"}), ("max_slots_eq", {"GW_BIT_MAX_SLOTS": "n_slots"}),
                ("max_slots_less", {"GW_BIT_MAX_SLOTS": "n_slots - 1"})]


def _run_device(torch, g, inp, B, stream=None):
    """the device entry point on B sets, outputs pre-filled with 0xFF bytes; returns (out, flags) tensors (not synchronized)"""
    d_in = torch.from_numpy(np.ascontiguousarray(inp[:B])).cuda()
    d_out = torch.full((B, g.n_witness * 32), 0xFF, dtype=torch.uint8, device="cuda")
    d_flags = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    g.calc_witness_batch_device(0, d_in.data_ptr(), B, d_out.data_ptr(), d_flags.data_ptr(), stream=stream)
    return d_in, d_out, d_flags


@pytest.mark.parametrize("variant", [name for name, _ in BIT_VARIANTS])
def test_corpus_under_bit_variant(cwc, monkeypatch, capfd, dev, corpus, variant):
    """every graph of the corpus under one bit-plan option, at B = 1, 2, 31, 32, 33, 65 and 1029 through the device entry
    point: the device compiled the simulator's plan, picked the launch the heuristic says, and got every row and flag right;
    the launches of the variant reach every step-residue class they are meant to"""
    torch = pytest.importorskip("torch")
    env0 = dict(BIT_VARIANTS)[variant]
    seen = {"single": set(), "ring": set(), "reg": set()}
    chunks = {"single": set(), "ring": set()}
    reg_long = False
    for case in corpus:
        sim = case.bits[env0.get("GW_BIT_MERGE") != "0"]
        env = dict(env0)
        eligible = True
        if "GW_BIT_MAX_SLOTS" in env:
            n_slots = sim.info["n_slots"]
            env["GW_BIT_MAX_SLOTS"] = str(n_slots if variant == "max_slots_eq" else n_slots - 1)
            eligible = variant == "max_slots_eq"
        _set_env(monkeypatch, env)
        g = cwc.Graph(case.data)
        assert g.info["bit_eligible"] == int(eligible), (case.name, variant)
        if eligible:
            for k_dev, k_sim in (("bit_steps", "n_steps"), ("bit_luts", "n_luts"), ("bit_wide", "n_wide")):
                assert g.info[k_dev] == sim.info[k_sim], (case.name, variant, k_dev)
        capfd.readouterr()
        for B in BATCHES:
            if B > len(case.inp):
                continue
            _, d_out, d_flags = _run_device(torch, g, case.inp, B)
            torch.cuda.synchronize()
            tr = _traces(capfd)
            takes_bit = eligible and B >= int(env.get("GW_BIT_MIN_SETS", 1))
            if not takes_bit:
                assert tr == [], (case.name, variant, B, tr)
            else:
                want = expected_launch(sim.info, B, dev, env)
                assert tr == [want], (case.name, variant, B, tr, want)
                n_steps = sim.info["n_steps"]
                seen[want[0]].add((n_steps - 1) % 16)
                if want[0] in chunks:
                    chunks[want[0]].add(min(util.bit_chunks(n_steps, util.BIT_CHUNK_SINGLE if want[0] == "single" else util.BIT_CHUNK_BATCH), 7))
                reg_long |= want[0] == "reg" and n_steps >= 128
            case.check(d_out.cpu().numpy(), d_flags.cpu().numpy().view(np.uint32), B, variant)
        assert _bit_eligible(cwc, g) == int(eligible), (case.name, variant, "speculation dropped")
        g.close()
    if variant in ("defaults", "ring_1", "ring_0", "merge_0", "max_slots_eq"):
        assert seen["single"] == set(range(16)) and {1, 2, 3, 4} <= chunks["single"], (variant, seen["single"], chunks["single"])
    if variant == "ring_1":
        assert {r % 8 for r in seen["ring"]} == set(range(8)) and {1, 2, 3, 4, 7} <= chunks["ring"], (seen["ring"], chunks["ring"])
    if variant in ("ring_0", "defaults"):
        assert {r % 4 for r in seen["reg"]} == set(range(4)), seen["reg"]
    if variant == "ring_0":
        assert reg_long, "the register variant never ran a program of >= 128 steps"
    if variant == "defaults":
        assert seen["ring"], "the ring variant never ran"
    if variant == "min_sets_33":
        assert not seen["single"] and seen["ring"] | seen["reg"]


@pytest.fixture(scope="module")
def narrow_graphs():
    """Boolean graphs with a narrow witness for the wide launches: a short program (< 128 steps) and a long one"""
    rnd = random.Random(31337)
    out = {}
    while len(out) < 2:
        nodes, wit, imap = boolean_graph(rnd, n_inputs=24, n_gates=rnd.choice([90, 300]))
        data = po.serialize_graph(nodes, wit, imap)
        s = util.BitSimGraph(data)
        if not s.info["eligible"] or not s.info["n_luts"] or len(wit) > 400:
            continue
        key = "long" if s.info["n_steps"] >= 128 else "short"
        out.setdefault(key, (data, s))
    return out


def _wide_rows(rng, B, n_in, con):
    inp = np.zeros((B, n_in, 32), dtype=np.uint8)
    inp[:, 0, 0] = 1
    inp[:, 1:, 0] = rng.integers(0, 2, size=(B, n_in - 1), dtype=np.uint8)
    bad = sorted(set(rng.choice(B, size=40, replace=False).tolist()) | {B - 1})
    for k, b in enumerate(bad):
        inp[b, con[k % len(con)]] = np.frombuffer(BAD_VALUES[k % len(BAD_VALUES)].to_bytes(32, "little"), dtype=np.uint8)
    return inp, bad


@pytest.mark.parametrize("which", ["short", "long"])
def test_wide_launches(cwc, monkeypatch, capfd, dev, narrow_graphs, which):
    """B = 2 * wpb * SMs * 32 +- 32 sets for wpb = 2, 4, 8 (warps per CTA from 1 to 8, a last CTA whose tail warps exit) under
    GW_BIT_RING unset, 0 and 1 and GW_BIT_WARPS=3: the whole batch byte for byte equal to the generic kernel's (GW_BITSLICE=0),
    and the oracle on rows 32 g and 32 g + 31 of every 37th group, every bad set and the last group"""
    torch = pytest.importorskip("torch")
    data, sim = narrow_graphs[which]
    con = contract_inputs(data)[0]
    rng = np.random.default_rng(17 if which == "short" else 18)
    Bs = [2 * w * dev["sms"] * 32 + d for w in (2, 4, 8) for d in (-32, 32)]
    inp, bad = _wide_rows(rng, max(Bs), sim.I, con)
    _set_env(monkeypatch, {"GW_BITSLICE": "0"})
    ref = cwc.Graph(data)
    shapes = set()
    for B in Bs:
        d_in, want_out, want_flags = _run_device(torch, ref, inp, B)
        torch.cuda.synchronize()
        groups = (B + 31) // 32
        check = sorted({r for g in range(0, groups, 37) for r in (32 * g, 32 * g + 31)} | {b for b in bad if b < B} | set(range(32 * (groups - 1), B)))
        check = [r for r in check if r < B]
        want = cref.CGraph(data).evaluate_batch(inp[check], os.cpu_count() or 4)
        got = want_out.cpu().numpy().reshape(B, -1, 32)[check]
        assert (got == want).all(), f"{which}: generic kernel differs from the oracle at B={B}"
        for name, env in (("auto", {}), ("ring_0", {"GW_BIT_RING": "0"}), ("ring_1", {"GW_BIT_RING": "1"}), ("warps_3", {"GW_BIT_WARPS": "3"})):
            _set_env(monkeypatch, env)
            g = cwc.Graph(data)
            capfd.readouterr()
            _, d_out, d_flags = _run_device(torch, g, inp, B)
            torch.cuda.synchronize()
            tr = _traces(capfd)
            exp = expected_launch(sim.info, B, dev, env)
            assert tr == [exp], (which, name, B, tr, exp)
            shapes.add(exp[:2])
            assert torch.equal(d_out, want_out), f"{which} {name} B={B}: witness differs from the generic kernel's"
            assert torch.equal(d_flags, want_flags), f"{which} {name} B={B}: flags differ from the generic kernel's"
            g.close()
        del d_in, want_out, want_flags
    ref.close()
    assert {w for v, w in shapes if v == "ring"} >= {1, 2, 3, 4, 7, 8}, shapes
    assert {w for v, w in shapes if v == "reg"} >= {1, 2, 3, 4, 7, 8}, shapes


def _json(imap, row):
    (name, (off, ln)), = imap.items()
    return json.dumps({name: [str(v % M) for v in row[off:off + ln]]})


CAP_POINTS = ("single_max", "single_past", "optin", "optin_past")
# (k, n_in) of util.bit_chain_graph with a given number of plane slots (the simulator's slot allocation is not linear in k):
# the four points of a B200 (232 448 bytes of opt-in shared memory); the one past the opt-in limit has 58 114 slots
CAP_HINTS = {51960: (51787, 352), 51961: (51800, 351), 58112: (58015, 350), 58113: (58016, 350)}


def _chain_for(target, exact):
    """(k, n_in) of a chain graph with `target` plane slots (exact) or a few more; a short walk over k from an estimate where
    the hints do not apply"""
    def n_slots(k, n_in):
        return util.BitSimGraph(po.serialize_graph(*util.bit_chain_graph(k, n_in)), max_slots=0xFFFE).info["n_slots"]
    ok = (lambda n: n == target) if exact else (lambda n: target <= n <= target + 2)
    if target in CAP_HINTS and ok(n_slots(*CAP_HINTS[target])):
        return CAP_HINTS[target]
    for n_in in (350, 351, 352, 353):
        k, seen = target - n_in + 190, {}
        while k not in seen and len(seen) < 12:
            seen[k] = n = n_slots(k, n_in)
            if ok(n):
                return k, n_in
            k += target - n if abs(target - n) > 2 else (1 if n < target else -1)
    raise AssertionError(f"no chain graph has {target} plane slots")


@pytest.mark.parametrize("point", CAP_POINTS)
def test_plane_file_capacity(cwc, monkeypatch, capfd, dev, point):
    """a graph whose plane file is the largest that still fits the single-set ring, one slot past it (B = 1 takes the batch
    kernels), exactly the device's opt-in shared memory (register variant only), and one slot past that, where the device
    is left to the generic kernels: the batch, latency and drop-in entry points all return the oracle's witness"""
    torch = pytest.importorskip("torch")
    smem = dev["smem"]
    # plane file + 3 mbarriers + 3 chunks of 16 LUT headers (single ring); the plane file alone (register variant)
    target = (smem - 32 - 3 * 16 * 512) // 4 if point.startswith("single") else smem // 4
    target += point.endswith("_past")
    k, n_in = _chain_for(target, exact=not point.endswith("_past"))
    nodes, wit, imap = util.bit_chain_graph(k, n_in)
    data = po.serialize_graph(nodes, wit, imap)
    sim = util.BitSimGraph(data, max_slots=0xFFFE)
    planes_b = (sim.info["n_slots"] * 4 + 15) & ~15
    assert (planes_b + 32 + 3 * 16 * 512 <= smem) == (point == "single_max")
    assert (planes_b <= smem) == (point != "optin_past")
    rnd = random.Random(5)
    rows = [[1] + [rnd.randrange(2) for _ in range(n_in)] for _ in range(4)]
    rows[2][7] = 2                                     # off the contract: the generic plan
    case = Case(f"chain_{k}", data, rows)
    # GW_THREADS=32: the generic plan of tens of thousands of live values spills them per resident thread (sms x 32 threads)
    base = {"GW_BIT_MAX_SLOTS": "65534", "GW_THREADS": "32"}
    for env in (base, dict(base, GW_BIT_RING="0")):
        _set_env(monkeypatch, env)
        g = cwc.Graph(data)
        assert g.info["bit_eligible"] == 1 and g.info["bit_steps"] == sim.info["n_steps"]
        capfd.readouterr()
        for B in (1, 4):
            _, d_out, d_flags = _run_device(torch, g, case.inp, B)
            torch.cuda.synchronize()
            tr = _traces(capfd)
            if point == "optin_past":
                assert tr == [], tr
            else:
                assert tr == [expected_launch(sim.info, B, dev, env)], (point, B, tr)
                if point == "single_past" and B == 1:
                    assert tr[0][0] == ("reg" if env.get("GW_BIT_RING") == "0" else "ring")
            case.check(d_out.cpu().numpy(), d_flags.cpu().numpy().view(np.uint32), B, f"{point} {env}")
        for b in range(len(rows)):
            try:
                out, flags = g.calc_witness_latency(case.inp[b], want_flags=True)
            except cwc.WitnessCalcError as e:          # the generic latency plan has no room for so many live values
                assert (b == 2 or point == "optin_past") and "too wide" in str(e), (point, b, str(e))
                continue
            assert (out == case.want[b]).all(), f"{point} latency row {b}"
            assert flags == case.flags[b]
        g.close()
    _set_env(monkeypatch, base)
    got = cwc.calc_witness_wtns(_json(imap, rows[1]), data)
    assert got == po.wtns_from_witness(util.unpack_u256(case.want[1].tobytes())), f"{point}: drop-in entry point"


def _sequence_rows(rnd, case_data, want_len=12):
    """good, bad, good rows (bad: rows 2 and 5) in an order where every witness position that varies changes between two
    consecutive rows somewhere (util.assert_rows_expose_stores): the latency entry point reuses one output buffer"""
    for attempt in range(40):
        n = want_len + attempt
        rows = corpus_rows(rnd, case_data, n, [2, 5])
        want = cref.CGraph(case_data).evaluate_batch(_pack(rows), 4)
        try:
            util.assert_rows_expose_stores("sequence", want)
            return rows
        except AssertionError:
            continue
    raise AssertionError("no row sequence exposes every store")


def test_single_witness_sequences(cwc, monkeypatch, capfd, corpus):
    """graphs whose programs fill 1 .. 4 chunks of the single-set ring: good, bad, good rows through the latency entry point
    (the single-set kernel; a bad set takes the generic latency plan), the drop-in entry point and a batch of one"""
    rnd = random.Random(4711)
    chunks = set()
    for case in corpus:
        sim = case.bits[True]
        n_ch = util.bit_chunks(sim.info["n_steps"], util.BIT_CHUNK_SINGLE)
        if not sim.info["n_luts"] or n_ch > 4 or n_ch in chunks:
            continue
        chunks.add(n_ch)
        seq = Case(case.name, case.data, _sequence_rows(rnd, case.data))
        nodes, wit, imap = po.deserialize_graph(case.data)
        _set_env(monkeypatch, {})
        g = cwc.Graph(case.data)
        capfd.readouterr()
        for b in range(len(seq.inp)):
            out, flags = g.calc_witness_latency(seq.inp[b], want_flags=True)
            assert _traces(capfd) == [("single", 1, 1, 1)], (case.name, b)
            assert (out == seq.want[b]).all(), f"{case.name} latency row {b}"
            assert flags == seq.flags[b], f"{case.name} latency row {b}: flags"
            out1, fl1 = g.calc_witness_batch(seq.inp[b:b + 1], want_flags=True)
            assert _traces(capfd) == [("single", 1, 1, 1)], (case.name, "batch of one", b)
            assert (out1[0] == seq.want[b]).all() and fl1[0] == seq.flags[b], f"{case.name} batch of one, row {b}"
            js = _json(imap, util.unpack_u256(seq.inp[b].tobytes()))
            buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(js))
            want = cref.CGraph(case.data).evaluate_batch(_pack([buf]), 1)[0]
            assert cwc.calc_witness_wtns(js, case.data) == po.wtns_from_witness(util.unpack_u256(want.tobytes())), (case.name, "drop-in", b)
            capfd.readouterr()
        g.close()
    assert chunks == {1, 2, 3, 4}, chunks


def _device_check(case, d_out, d_flags, B, what):
    case.check(d_out.cpu().numpy(), d_flags.cpu().numpy().view(np.uint32), B, what)


def test_speculation_drop(cwc, monkeypatch, capfd, narrow_graphs):
    """the bit path is dropped for a graph after a launch of >= 64 sets of which more than half broke the contract, and only
    then: 64 sets with 33 bad drop it, 64 with 32 bad and 63 all bad keep it; every result is exact, also the latency calls
    after the drop"""
    torch = pytest.importorskip("torch")
    data, sim = narrow_graphs["long"]
    rnd = random.Random(64)
    for n_sets, n_bad, drops in ((64, 33, True), (64, 32, False), (63, 63, False)):
        bad = rnd.sample(range(n_sets), n_bad)
        rows = corpus_rows(rnd, data, n_sets, bad)
        case = Case(f"drop_{n_sets}_{n_bad}", data, rows)
        _set_env(monkeypatch, {})
        g = cwc.Graph(data)
        capfd.readouterr()
        _, d_out, d_flags = _run_device(torch, g, case.inp, n_sets)
        torch.cuda.synchronize()
        assert len(_traces(capfd)) == 1
        _device_check(case, d_out, d_flags, n_sets, "first launch")
        assert _bit_eligible(cwc, g) == 1, "the count is looked at on the next launch"
        good = [b for b in range(n_sets) if b not in bad] or [0]
        _, d_out, d_flags = _run_device(torch, g, case.inp[good], len(good))
        torch.cuda.synchronize()
        case.want, case.flags = case.want[good], case.flags[good]
        _device_check(case, d_out, d_flags, len(good), "second launch")
        assert _bit_eligible(cwc, g) == int(not drops), (n_sets, n_bad)
        capfd.readouterr()
        _, d_out, d_flags = _run_device(torch, g, case.inp[good], len(good))
        torch.cuda.synchronize()
        assert (len(_traces(capfd)) == 1) != drops, (n_sets, n_bad)
        _device_check(case, d_out, d_flags, len(good), "third launch")
        full = Case(case.name, data, rows)
        for b in (good[0], bad[0]):
            out, flags = g.calc_witness_latency(full.inp[b], want_flags=True)
            assert (out == full.want[b]).all() and flags == full.flags[b], (case.name, "latency", b)
        g.close()


def test_streams_and_shared_scratch(cwc, monkeypatch, capfd, narrow_graphs):
    """the per-device scratch of the bit path (planes, ok words, bad list and count) shared by calls on different streams: a
    device batch on a side stream left running, a latency call, a device batch of more groups on another stream (the scratch
    is reallocated), and a host call cut into 4 chunks on the engine's two streams; every result exact"""
    torch = pytest.importorskip("torch")
    data, sim = narrow_graphs["long"]
    rnd = random.Random(99)
    chunk = (1 << 20) // (32 * (sim.I + sim.W))          # sets per chunk of the host call under GW_CHUNK_MB=1
    n1, n3, n4 = 100, 3000, 3 * chunk + 5
    rows = corpus_rows(rnd, data, n1 + 1 + n3 + n4, [3, 40, 77, n1 + 1 + 5, n1 + 1 + 2000, n1 + 1 + n3 + 1, n1 + 1 + n3 + 2, n1 + 1 + n3 + 30])
    parts = {"first": slice(0, n1), "latency": slice(n1, n1 + 1), "larger": slice(n1 + 1, n1 + 1 + n3), "host": slice(n1 + 1 + n3, None)}
    cases = {k: Case(k, data, rows[s]) for k, s in parts.items()}
    _set_env(monkeypatch, {"GW_CHUNK_MB": "1"})
    g = cwc.Graph(data)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    capfd.readouterr()
    d_in1 = torch.from_numpy(cases["first"].inp.copy()).cuda()
    d_out1 = torch.full((n1, g.n_witness * 32), 0xFF, dtype=torch.uint8, device="cuda")
    d_fl1 = torch.full((n1,), -1, dtype=torch.int32, device="cuda")
    d_in3 = torch.from_numpy(cases["larger"].inp.copy()).cuda()
    d_out3 = torch.full((n3, g.n_witness * 32), 0xFF, dtype=torch.uint8, device="cuda")
    d_fl3 = torch.full((n3,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    g.calc_witness_batch_device(0, d_in1.data_ptr(), n1, d_out1.data_ptr(), d_fl1.data_ptr(), stream=s1.cuda_stream)
    out_l, fl_l = g.calc_witness_latency(cases["latency"].inp[0], want_flags=True)
    g.calc_witness_batch_device(0, d_in3.data_ptr(), n3, d_out3.data_ptr(), d_fl3.data_ptr(), stream=s2.cuda_stream)
    out_h, fl_h = g.calc_witness_batch(cases["host"].inp, want_flags=True)
    torch.cuda.synchronize()
    err = capfd.readouterr().err
    kinds = [m.group(1) for m in TRACE.finditer(err)]
    assert len(kinds) == 2 + 1 + 4 and kinds[1] == "single", kinds
    m = re.search(r"\[gw trace\] device 0: (\d+) sets, chunk (\d+)", err)
    assert m and int(m.group(1)) == n4 and int(m.group(2)) == chunk, m and m.group(0)
    cases["first"].check(d_out1.cpu().numpy(), d_fl1.cpu().numpy().view(np.uint32), n1, "side stream")
    cases["latency"].check(out_l[None], [fl_l], 1, "latency between batches")
    cases["larger"].check(d_out3.cpu().numpy(), d_fl3.cpu().numpy().view(np.uint32), n3, "second stream, reallocated scratch")
    cases["host"].check(out_h, fl_h, n4, "host call in one-set chunks")
    assert _bit_eligible(cwc, g) == 1
    g.close()
