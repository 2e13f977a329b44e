"""The throughput interpreter (eval_batch_kernel) under every plan option and launch shape, row by row against the C oracle.

The plan compiler is checked on the host simulator (tests/test_plan_sim.py); the device loop has code of its own for the
instruction ring, the OP_DOT term decoding, the hot / __ldg constant split, the spill areas and the persistent tile loop.
Here the same corpus (test_plan_sim.matrix_corpus) runs on the GPU under each option of util.PLAN_VARIANTS, and one batch
runs at launch shapes of one CTA, one wave and several tiles per CTA through both entry points.  Every witness value must
equal the oracle's and every per-set flag the simulator's; util.assert_plan_coverage says the programs reach the paths
they are there for."""
import importlib
import os
import random
import re

import numpy as np
import pytest

from oracle import cref
from tests import util
from tests.test_plan_sim import matrix_corpus
from tests.util import po

pytestmark = pytest.mark.gpu

ENV_KEYS = ("GW_DIV_BATCH", "GW_FUSE_DOT", "GW_MAX_TERMS", "GW_NARROW", "GW_FUSE_POW5", "GW_REGS", "GW_HOT_CONSTS", "GW_THREADS",
            "GW_CHUNK_MB", "GW_TRACE_HOST", "GW_BITSLICE")
LAUNCH_THREADS = 32          # GW_THREADS of the launch-shape tests: a wave is sms x 32 sets, so several waves are cheap


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


def _set_env(monkeypatch, env, n_consts=0):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("GW_BITSLICE", "0")          # the generic kernel for every graph (Boolean ones included)
    for k, v in env.items():
        monkeypatch.setenv(k, str(n_consts // 2) if v == "half" else v)


def _pack(rows):
    return np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32)


class Case:
    """a graph, an input batch, the oracle's witness rows and the simulator's per-set flags"""

    def __init__(self, name, nodes, wit, imap, rows):
        self.name, self.data = name, po.serialize_graph(nodes, wit, imap)
        self.inp = _pack(rows)
        self.want = cref.CGraph(self.data).evaluate_batch(self.inp, os.cpu_count() or 4)
        sim = util.SimGraph(self.data, **util.sim_options({}))
        self.flags = np.array([sim.eval(r)[1] for r in rows], dtype=np.uint32)
        self.n_consts = sim.info["n_consts"]

    def check(self, out, flags, B=None, what=""):
        B = len(self.inp) if B is None else B
        bad = np.nonzero((out.reshape(B, -1) != self.want[:B].reshape(B, -1)).any(axis=1))[0]
        assert len(bad) == 0, f"{self.name} {what}: {len(bad)} wrong witness rows of {B}, first {bad[:8].tolist()}"
        badf = np.nonzero(flags[:B] != self.flags[:B])[0]
        assert len(badf) == 0, f"{self.name} {what}: wrong flags in rows {badf[:8].tolist()}: {flags[badf[:4]]} != {self.flags[badf[:4]]}"


@pytest.fixture(scope="module")
def corpus():
    return [Case(*c) for c in matrix_corpus()]


@pytest.mark.parametrize("variant", [name for name, _ in util.PLAN_VARIANTS])
def test_corpus_under_plan_option(cwc, monkeypatch, corpus, variant):
    """every graph of the corpus under one option of the matrix: the device runs the program the simulator checks (same
    size, registers, OP_DOTs, inversions) and gets every row right"""
    env = dict(util.PLAN_VARIANTS)[variant]
    cov = None
    for case in corpus:
        _set_env(monkeypatch, env, case.n_consts)
        sim = util.SimGraph(case.data, **util.sim_options(env))
        g = cwc.Graph(case.data)
        for k_dev, k_sim in (("n_slots", "slots"), ("n_regs", "n_regs"), ("n_dot", "n_dot"), ("n_inversions", "inversions")):
            assert g.info[k_dev] == sim.info[k_sim], (case.name, k_dev)
        out, flags = g.calc_witness_batch(case.inp, want_flags=True)
        case.check(out, flags, what=variant)
        c = util.plan_coverage(sim.code())
        cov = c if cov is None else util.merge_coverage(cov, c)
        g.close()
    util.assert_plan_coverage(cov, util.VARIANT_FEATURES.get(variant, ()))


def _flag_graph(rnd):
    """a random graph whose per-set flags depend on the row (Shl overflow, bitwise results equal to M): no Pow, Id, Lnot
    or Bnot, which flag every row"""
    return util.random_graph(rnd, n_ops=400, ops=[op for op in range(20) if op != po.DUO["Pow"]], uno_ext=False)


@pytest.fixture(scope="module")
def shape_cases(cwc):
    torch = pytest.importorskip("torch")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    wave = sms * LAUNCH_THREADS
    n_rows = 3 * wave + 77
    rnd = random.Random(606)
    cases = []
    from tests.test_plan_sim import _narrow_graph
    for name, (nodes, wit, imap) in (("flags", _flag_graph(rnd)), ("narrow", _narrow_graph(rnd, n_ops=250))):
        base = [util.matrix_row(rnd, 6) for _ in range(509)]
        rows = [base[(b * 7) % 509] if b % 3 else util.matrix_row(rnd, 6) for b in range(n_rows)]
        cases.append(Case(name, nodes, wit, imap, rows))
    assert len(set(cases[0].flags.tolist())) > 2, "the flag graph must flag some rows and not others"
    return wave, cases


LAUNCH_VARIANTS = [("threads_32", {}), ("regs_4", {"GW_REGS": "4"}), ("max_terms_16", {"GW_MAX_TERMS": "16", "GW_REGS": "24"}),
                   ("hot_0", {"GW_HOT_CONSTS": "0"})]


@pytest.mark.parametrize("entry", ["device", "host"])
@pytest.mark.parametrize("variant", [name for name, _ in LAUNCH_VARIANTS])
def test_launch_shapes(cwc, monkeypatch, capfd, shape_cases, entry, variant):
    """batches of 1, 31 and 33 sets, one wave -1 / +1, and three waves + 77 (every CTA runs several tiles: the tile loop
    re-stages the ring, resets the flags and reuses its spill slots), through the device entry point and through the host
    entry point cut into >= 3 chunks"""
    torch = pytest.importorskip("torch")
    wave, cases = shape_cases
    env = dict(LAUNCH_VARIANTS)[variant]
    for case in cases:
        _set_env(monkeypatch, dict(env, GW_THREADS=str(LAUNCH_THREADS)))
        g = cwc.Graph(case.data)
        if variant == "regs_4":
            assert g.info["n_spill"] > 0
        for B in (1, 31, 33, wave - 1, wave + 1, len(case.inp)):
            inp = case.inp[:B]
            if entry == "device":
                d_in = torch.from_numpy(inp.copy()).cuda()
                d_out = torch.empty((B, g.n_witness * 32), dtype=torch.uint8, device="cuda")
                d_flags = torch.full((B,), -1, dtype=torch.int32, device="cuda")
                g.calc_witness_batch_device(0, d_in.data_ptr(), B, d_out.data_ptr(), d_flags.data_ptr())
                torch.cuda.synchronize()
                out, flags = d_out.cpu().numpy(), d_flags.cpu().numpy().view(np.uint32)
            else:
                monkeypatch.setenv("GW_CHUNK_MB", "0" if B < 64 else "1")      # 0: one set per chunk
                monkeypatch.setenv("GW_TRACE_HOST", "1")
                capfd.readouterr()
                out, flags = g.calc_witness_batch(inp, want_flags=True)
                m = re.search(r"\[gw trace\] device 0: (\d+) sets, chunk (\d+)", capfd.readouterr().err)
                assert m and int(m.group(1)) == B
                assert -(-B // int(m.group(2))) >= min(B, 3), (B, m.group(0))
            case.check(out, flags, B, f"{variant} {entry} B={B}")
        g.close()


def test_one_batch_same_bytes_and_flags_under_every_option(cwc, monkeypatch, shape_cases):
    """one graph, one batch of a wave + 1 sets: every option of the matrix gives the same witness bytes and flags"""
    wave, cases = shape_cases
    case = cases[0]
    B = wave + 1
    first = None
    for name, env in util.PLAN_VARIANTS:
        _set_env(monkeypatch, env, case.n_consts)
        g = cwc.Graph(case.data)
        out, flags = g.calc_witness_batch(case.inp[:B], want_flags=True)
        g.close()
        case.check(out, flags, B, name)
        if first is None:
            first = (out, flags)
        assert (out == first[0]).all() and (flags == first[1]).all(), name


def test_two_gpu_shards(cwc, monkeypatch, shape_cases):
    """the host entry point sharded over two GPUs, every CTA of both running several tiles with a spilling plan"""
    if cwc.device_count() < 2:
        pytest.skip("one GPU visible")
    wave, cases = shape_cases
    for case in cases:
        _set_env(monkeypatch, {"GW_THREADS": str(LAUNCH_THREADS), "GW_REGS": "4"})
        g = cwc.Graph(case.data)
        out, flags = g.calc_witness_batch(case.inp, n_gpus=2, want_flags=True)
        g.close()
        case.check(out, flags, what="2 GPUs")
