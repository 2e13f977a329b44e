"""Latency-mode plan (csrc/plan.cpp: compile_latency_plan -- levels, warp assignment, packets, slow-warp jobs, chains,
split linear combinations) executed by the host simulator against the Python oracle.  The simulator models what the
kernel guarantees and nothing more: inside a level a lane sees only its own writes, and the slow-warp jobs run either as
early or as late as the protocol allows (tests/csrc/plan_host_sim.cpp).  No GPU needed."""
import random

import pytest

from tests import util
from tests.util import po

VARIANTS = [
    dict(),                                               # defaults: 7 main warps, 4 slow warps, chains, split dots
    dict(chain=False),
    dict(split_dot=False, chain=False),
    dict(fuse=False),                                     # one instruction per graph node
    dict(n_warps=1, n_slow_warps=1, slow_levels=1),       # everything serialised, readers right behind the long ops
    dict(n_warps=3, slow_levels=3, packet_slots=24),      # tiny packets: wide levels are cut into many physical levels
    dict(n_warps=12, n_slow_warps=2, slow_levels=40),
    # dataflow plan: per-warp packet streams with wait vectors; the simulator's `mode` picks the interleaving of the warps
    dict(dataflow=True),
    dict(dataflow=True, n_warps=1, n_slow_warps=1, slow_levels=1),
    dict(dataflow=True, n_warps=3, slow_levels=3, packet_slots=24),
    dict(dataflow=True, n_warps=8, n_slow_warps=4, fuse=False),
    dict(dataflow=True, split_dot=False),
    # S-box link rewrite forced (OP_POW4 + OP_MULADD, side sums written out), both plan kinds
    dict(dataflow=True, sbox_links=2),
    dict(sbox_links=2),
    dict(dataflow=True, sbox_links=0),
]


def _rows(rnd, n_in, n):
    return [[1] + [util.random_value(rnd) if rnd.random() < 0.8 else rnd.randrange(1 << 256) for _ in range(n_in)] for _ in range(n)]


@pytest.mark.parametrize("vi", range(len(VARIANTS)))
def test_random_graphs_all_ops(vi):
    rnd = random.Random(700 + vi)
    for t in range(12):
        nodes, wit, imap = util.random_graph(rnd, n_ops=300)
        g = util.SimGraph(po.serialize_graph(nodes, wit, imap), 12)
        for row in _rows(rnd, 6, 2):
            want = po.evaluate(nodes, row, wit, "circom")
            for mode in ((0, 1, 2, 3, 11) if VARIANTS[vi].get("dataflow") else (0, 1)):
                got, info = g.eval_latency(row, mode=mode, **VARIANTS[vi])
                assert got == want, (vi, t, mode)


def test_division_chains_and_parallel_divisions():
    """long ops: a dependent chain (every Div feeds the next) next to a batch of independent ones, read immediately"""
    rnd = random.Random(11)
    nodes = [(po.K_INPUT, i) for i in range(7)] + [(po.K_CONST, 3)]
    acc = 1
    for k in range(12):
        nodes.append((po.K_DUO, po.DUO["Div"], acc, 1 + (k % 6)))      # chain
        acc = len(nodes) - 1
        nodes.append((po.K_DUO, po.DUO["Add"], acc, 7))
        acc = len(nodes) - 1
    par = []
    for k in range(40):                                                    # 40 independent divisions: two 32-lane jobs
        nodes.append((po.K_DUO, po.DUO["Div"], 1 + k % 6, 1 + (k + 1) % 6))
        par.append(len(nodes) - 1)
    for k in par:
        nodes.append((po.K_DUO, po.DUO["Mul"], k, acc))
    for name in ("Idiv", "Mod", "Pow"):
        nodes.append((po.K_DUO, po.DUO[name], 2, 7))
    wit = [0] + list(range(8, len(nodes)))
    g = util.SimGraph(po.serialize_graph(nodes, wit, {"x": (1, 6)}), 12)
    for row in _rows(rnd, 6, 3) + [[1, 0, 0, 0, 0, 0, 0]]:              # division by zero -> 0 (graph.rs:109)
        want = po.evaluate(nodes, row, wit, "circom")
        for kw in VARIANTS:
            for mode in ((0, 1, 2, 7) if kw.get("dataflow") else (0, 1)):
                got, info = g.eval_latency(row, mode=mode, **kw)
                assert got == want, (kw, mode)


def test_edge_graphs():
    rnd = random.Random(5)
    cases = [([(po.K_INPUT, 0)], [], {}, 0),
             ([(po.K_INPUT, 0), (po.K_CONST, 7)], [1, 1, 0, 1], {}, 0),
             ([(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, 5), (po.K_CONST, 9), (po.K_TRES, 0, 1, 2, 3), (po.K_TRES, 0, 2, 1, 4)],
              [0, 4, 5, 4], {"x": (1, 1)}, 1)]
    for nodes, wit, imap, n_in in cases:
        g = util.SimGraph(po.serialize_graph(nodes, wit, imap), 8)
        for row in _rows(rnd, n_in, 2):
            for mode in (0, 1):
                assert g.eval_latency(row, mode=mode)[0] == po.evaluate(nodes, row, wit, "circom")
                assert g.eval_latency(row, mode=mode, dataflow=True)[0] == po.evaluate(nodes, row, wit, "circom")


@pytest.mark.parametrize("name", ["circuit5_poseidon", "circuit6_num2bits", "circuit11_key_expansion", "circuit8_sha256_512", "circuit9_authV2"])
def test_golden_circuits(name):
    data = util.golden_graph(name)
    nodes, wit, imap = po.deserialize_graph(data)
    buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs(name)))
    want = po.parse_wtns(util.golden_wtns(name))
    g = util.SimGraph(data, 12)
    for kw in (dict(), dict(chain=False), dict(n_warps=2, slow_levels=2, packet_slots=40), dict(dataflow=True), dict(dataflow=True, n_warps=8),
               dict(dataflow=True, n_warps=2, slow_levels=2, packet_slots=48)):
        for mode in ((0, 1, 5) if kw.get("dataflow") else (0, 1)):
            got, info = g.eval_latency(buf, mode=mode, **kw)
            assert got == want, (name, kw, mode)
    got, info = g.eval_latency(buf)
    if name in ("circuit5_poseidon", "circuit9_authV2"):
        # S-boxes are one OP_POW5 (or a lane chain), linear combinations are split into an early and a late part:
        # well under half the levels of the one-instruction-per-node schedule
        assert info["n_split"] > 0
        assert 2 * info["n_levels"] < g.eval_latency(buf, fuse=False, chain=False)[1]["n_levels"]
    if name == "circuit8_sha256_512":
        assert info["n_chained"] == 0                             # the cost model keeps lane parallelism for bit-level graphs


def test_poseidon_like_graphs():
    """random graphs with Poseidon's shapes (tests/util.py: poseidon_like_graph): OP_POW5, the straight-line OP_DOT shapes,
    Mul(const, x + c) folding, chains, split linear combinations, divisions on the slow warps"""
    for seed in range(120):
        rnd = random.Random(3000 + seed)
        nodes, wit, imap = util.poseidon_like_graph(rnd, rnd.choice([2, 3, 5]), rnd.choice([3, 8, 20]))
        g = util.SimGraph(po.serialize_graph(nodes, wit, imap), 12)
        row = _rows(rnd, 6, 1)[0]
        want = po.evaluate(nodes, row, wit, "circom")
        for mode in (0, 1, 2 + seed):
            assert g.eval_latency(row, mode=mode, **VARIANTS[seed % len(VARIANTS)])[0] == want, (seed, mode)


def test_sbox_link_rewrite_on_poseidon_graphs():
    """S*x^5 on the path from one S-box to the next becomes (S*x)*x^4 (plan.cpp: rewrite_sbox_links): every partial round
    of the circomlib Poseidons is rewritten, values unchanged; left to itself the compiler keeps the rewrite for a lone
    Poseidon and drops it for authV2 (timing model)."""
    for name, rounds in (("circuit5_poseidon", 57), ("poseidon2", 57), ("circuit7_poseidon4", 60)):
        data = util.golden_graph(name)
        nodes, wit, imap = po.deserialize_graph(data)
        buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs(name)))
        want = po.parse_wtns(util.golden_wtns(name))
        g = util.SimGraph(data, 12)
        for kw in (dict(dataflow=True, sbox_links=2), dict(sbox_links=2), dict(dataflow=True)):
            for mode in (0, 1, 4):
                got, info = g.eval_latency(buf, mode=mode, **kw)
                assert got == want, (name, kw, mode)
            assert info["n_sbox_links"] >= rounds, (name, kw, info)
    g = util.SimGraph(util.golden_graph("circuit9_authV2"), 12)
    data = util.golden_graph("circuit9_authV2")
    nodes, wit, imap = po.deserialize_graph(data)
    buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs("circuit9_authV2")))
    want = po.parse_wtns(util.golden_wtns("circuit9_authV2"))
    got, info = g.eval_latency(buf, mode=2, dataflow=True, sbox_links=2)
    assert got == want and info["n_sbox_links"] > 4000
    got, info = g.eval_latency(buf, mode=2, dataflow=True)
    assert got == want and info["n_sbox_links"] == 0


@pytest.mark.parametrize("variant", [name for name, _ in util.LATENCY_VARIANTS])
def test_latency_matrix_corpus(variant):
    """every graph of the latency corpus (util.latency_corpus) under one option of the latency matrix, on the simulator:
    every value against the C oracle, the status against the throughput plan's, the slow-warp jobs or the warp interleaving
    at both extremes (and one pseudo-random interleaving of the dataflow plan); and the corpus reaches what it is there for
    (util.assert_latency_coverage).  A graph whose live values do not fit the value file must be refused as too wide."""
    import numpy as np
    from oracle import cref
    opts = util.latency_sim_options(dict(util.LATENCY_VARIANTS)[variant])
    modes = (0, 1, 17) if opts["dataflow"] else (0, 1)
    cov = None
    for name, nodes, wit, imap, rows in util.latency_corpus():
        data = po.serialize_graph(nodes, wit, imap)
        g = util.SimGraph(data, **util.sim_options({}))
        want = cref.CGraph(data).evaluate_batch(np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32), 4)
        util.assert_rows_expose_stores(name, want)
        for b, r in enumerate(rows):
            status = g.eval(r)[1]
            for mode in modes:
                try:
                    got, info, c = g.eval_latency(r, mode=mode, coverage=True, **opts)
                except ValueError as e:
                    assert "too wide" in str(e) and name == "const_heavy" and not opts["fuse"], (name, str(e))
                    break
                assert got == util.unpack_u256(want[b].tobytes()), (name, b, mode)
                assert info["status"] == status, (name, b, mode)
                cov = c if cov is None else util.merge_coverage(cov, c)
    util.assert_latency_coverage(cov, util.LATENCY_VARIANT_FEATURES[variant])
