"""The single-witness latency kernels (eval_dataflow_kernel, and eval_latency_kernel under GW_LAT_MODE=level) under every
latency plan option, at the capacity of the shared-memory value file and in the call sequences a user makes, row by row
against the C oracle.

The plan compiler is checked on the host simulator (tests/test_latency_plan.py); the kernels have code of their own for the
packet rings (TMA copies completing on mbarriers), the level barrier and the slow-warp job protocol, the dataflow wait vectors
and progress counters, the straight-line and generic OP_DOT paths, packet-relative constants and the slow-warp constants read
from global memory.  Here util.latency_corpus runs on the GPU under each option of util.LATENCY_VARIANTS.  Every witness value
must equal the oracle's and every flag word the simulator's; consecutive rows give different witnesses, so a store the kernel
skips cannot hide behind the previous call's value in the reused output buffer; util.assert_latency_coverage says the plans
reach the paths they are there for."""
import importlib
import json
import os
import random

import numpy as np
import pytest

from oracle import cref
from tests import util
from tests.util import po

pytestmark = pytest.mark.gpu

ENV_KEYS = util.LATENCY_ENV_KEYS + ("GW_BITSLICE", "GW_DEVICE", "GW_REGS", "GW_FUSE_DOT", "GW_MAX_TERMS", "GW_DIV_BATCH", "GW_NARROW",
                                    "GW_FUSE_POW5", "GW_THREADS", "GW_HOT_CONSTS")


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


def _set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _pack(rows):
    return np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32)


class Case:
    """a graph, its input rows in call order, the oracle's witness rows and the throughput simulator's flag words"""

    def __init__(self, name, nodes, wit, imap, rows):
        self.name, self.nodes, self.wit, self.imap = name, nodes, wit, imap
        self.data = po.serialize_graph(nodes, wit, imap)
        self.rows = rows
        self.inp = _pack(rows)
        self.want = cref.CGraph(self.data).evaluate_batch(self.inp, os.cpu_count() or 4)
        util.assert_rows_expose_stores(name, self.want)
        self.sim = util.SimGraph(self.data, **util.sim_options({}))
        self.flags = [self.sim.eval(r)[1] for r in rows]

    def check(self, b, out, flags=None, what=""):
        bad = np.nonzero((out.reshape(-1, 32) != self.want[b].reshape(-1, 32)).any(axis=1))[0]
        assert len(bad) == 0, f"{self.name} {what} row {b}: {len(bad)} wrong witness positions, first {bad[:8].tolist()}"
        if flags is not None:
            assert flags == self.flags[b], f"{self.name} {what} row {b}: flags {flags:#x} != {self.flags[b]:#x}"


@pytest.fixture(scope="module")
def corpus():
    return [Case(*c) for c in util.latency_corpus()]


@pytest.mark.parametrize("variant", [name for name, _ in util.LATENCY_VARIANTS])
def test_corpus_under_latency_option(cwc, monkeypatch, corpus, variant):
    """every graph of the latency corpus under one option of the matrix: a fresh Graph (the options are read when its latency
    plan is first built), the rows in order through the latency entry point; a graph the simulator finds too wide for the
    value file must be refused as such"""
    env = dict(util.LATENCY_VARIANTS)[variant]
    opts = util.latency_sim_options(env)
    cov = None
    for case in corpus:
        _set_env(monkeypatch, env)
        try:
            _, _, c = case.sim.eval_latency(case.rows[0], coverage=True, **opts)
        except ValueError as e:
            assert "too wide" in str(e), (case.name, str(e))
            c = None
        g = cwc.Graph(case.data)
        if c is None:
            with pytest.raises(cwc.WitnessCalcError, match="too wide"):
                g.calc_witness_latency(case.inp[0])
            g.close()
            continue
        cov = c if cov is None else util.merge_coverage(cov, c)
        for b in range(len(case.rows)):
            out, flags = g.calc_witness_latency(case.inp[b], want_flags=True)
            case.check(b, out, flags, variant)
        g.close()
    util.assert_latency_coverage(cov, util.LATENCY_VARIANT_FEATURES[variant])


def _optin_smem():
    torch = pytest.importorskip("torch")
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _json(imap, row):
    (name, (off, ln)), = imap.items()
    return json.dumps({name: [str(v) for v in row[off:off + ln]]})


@pytest.mark.parametrize("mode", ["level", "dataflow", "dataflow_12"])
def test_value_file_capacity(cwc, monkeypatch, mode):
    """the widest graph whose value file fits the device's opt-in shared memory exactly (n_slots == max_slots: the value file
    ends where the packet rings begin and the launch asks for all of it) runs exact; one value more is refused as too wide
    by the latency entry point and computed by the drop-in entry point through the throughput kernel"""
    env = {"level": {"GW_LAT_MODE": "level"}, "dataflow": {}, "dataflow_12": {"GW_LAT_WARPS": "8", "GW_LAT_SLOW_WARPS": "4"}}[mode]
    env = dict(env, GW_LAT_BIT="0")
    optin = _optin_smem()
    opts = util.latency_sim_options(env, optin)
    cap = opts["max_slots"]
    rnd = random.Random(77)
    rows = [[1] + [util.random_value(rnd) for _ in range(6)] for _ in range(3)]

    def n_slots(k):
        try:
            return util.SimGraph(po.serialize_graph(*util.wide_live_graph(k)), 12).eval_latency(rows[0], **opts)[1]["n_slots"]
        except ValueError as e:
            assert "too wide" in str(e)
            return cap + 1
    lo, hi = 1, cap                       # n_slots(lo) <= cap < n_slots(hi)
    assert n_slots(lo) <= cap < n_slots(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if n_slots(mid) <= cap else (lo, mid)
    assert n_slots(lo) == cap, f"no graph fills the value file exactly: k = {lo} needs {n_slots(lo)} of {cap} slots"
    _set_env(monkeypatch, env)
    fit = Case(f"wide_live_{lo}", *util.wide_live_graph(lo), rows)
    g = cwc.Graph(fit.data)
    for b in range(len(rows)):
        out, flags = g.calc_witness_latency(fit.inp[b], want_flags=True)
        fit.check(b, out, flags, f"{mode} at capacity")
    g.close()
    wide = Case(f"wide_live_{lo + 1}", *util.wide_live_graph(lo + 1), rows)
    g = cwc.Graph(wide.data)
    with pytest.raises(cwc.WitnessCalcError, match="too wide"):
        g.calc_witness_latency(wide.inp[0])
    g.close()
    got = cwc.calc_witness_wtns(_json(wide.imap, rows[1]), wide.data)
    assert got == po.wtns_from_witness(util.unpack_u256(wide.want[1].tobytes())), f"{mode}: drop-in past capacity"


def _cases(corpus, names):
    by = {c.name: c for c in corpus}
    return [by[n] for n in names]


def test_call_sequences(cwc, monkeypatch, corpus):
    """latency, batch and latency calls on one Graph; two Graphs of the same bytes under the level and the dataflow plan,
    called alternately"""
    env = dict(util.LATENCY_VARIANTS)
    for case in _cases(corpus, ["poseidon_0", "div_group_33", "slow_const", "dot_shapes", "tern_muladd"]):
        _set_env(monkeypatch, env["df_defaults"])
        g = cwc.Graph(case.data)
        out, flags = g.calc_witness_latency(case.inp[0], want_flags=True)
        case.check(0, out, flags, "latency before batch")
        out, flags = g.calc_witness_batch(case.inp, want_flags=True)
        for b in range(len(case.rows)):
            case.check(b, out[b], int(flags[b]), "batch between latency calls")
        for b in range(1, len(case.rows)):
            out, flags = g.calc_witness_latency(case.inp[b], want_flags=True)
            case.check(b, out, flags, "latency after batch")
        g.close()
        graphs = []
        for v in ("level_defaults", "df_warps_12"):
            _set_env(monkeypatch, env[v])
            graphs.append(cwc.Graph(case.data))
            out, flags = graphs[-1].calc_witness_latency(case.inp[0], want_flags=True)       # builds the plan under v
            case.check(0, out, flags, v)
        _set_env(monkeypatch, {})
        for b in range(1, len(case.rows)):
            for v, g in zip(("level", "dataflow"), graphs):
                out, flags = g.calc_witness_latency(case.inp[b], want_flags=True)
                case.check(b, out, flags, f"alternating, {v}")
        for g in graphs:
            g.close()


def test_second_gpu_upload(cwc, monkeypatch, corpus):
    """one Graph on device 1 after device 0: the latency plan is uploaded per device"""
    if cwc.device_count() < 2:
        pytest.skip("one GPU visible")
    for v in ("df_defaults", "level_defaults"):
        for case in _cases(corpus, ["poseidon_1", "div_group_65", "dot_shapes"]):
            _set_env(monkeypatch, dict(util.LATENCY_VARIANTS)[v])
            g = cwc.Graph(case.data)
            for b in range(len(case.rows)):
                out, flags = g.calc_witness_latency(case.inp[b], device=b % 2, want_flags=True)
                case.check(b, out, flags, f"{v} device {b % 2}")
            g.close()


def test_drop_in_entry_point(cwc, monkeypatch, corpus):
    """gw_calc_witness (inputs JSON + graph bytes -> .wtns) under two latency options against the oracle's .wtns.  Parsed
    graphs are cached by content, so each option gets graphs of its own."""
    for v, names in (("level_defaults", ["dot_shapes", "slow_const", "poseidon_0", "chain_3"]),
                     ("df_warps_12", ["div_group_33", "tern_muladd", "lc_0", "chain_4"])):
        _set_env(monkeypatch, dict(util.LATENCY_VARIANTS)[v])
        for case in _cases(corpus, names):
            for b in range(len(case.rows)):
                js = _json(case.imap, [v % util.M for v in case.rows[b]])
                buf = po.build_input_buffer(case.nodes, case.imap, po.deserialize_inputs(js))
                want = cref.CGraph(case.data).evaluate_batch(_pack([buf]), 1)[0]
                got = cwc.calc_witness_wtns(js, case.data)
                assert got == po.wtns_from_witness(util.unpack_u256(want.tobytes())), (v, case.name, b)
