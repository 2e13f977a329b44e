"""Plan compiler (csrc/plan.cpp: liveness, constant table, register allocation, Belady spilling,
witness placement) executed by the host simulator with the same alu_exec() the kernel uses, against
the Python oracle.  No GPU needed."""
import random

import numpy as np
import pytest

from tests import util
from tests.util import po


def _check(nodes, wit, imap, n_regs, rnd, n_rows=3, n_in=6):
    g = util.SimGraph(po.serialize_graph(nodes, wit, imap), n_regs)
    for _ in range(n_rows):
        inp = [1] + [util.random_value(rnd) if rnd.random() < 0.8 else rnd.randrange(1 << 256) for _ in range(n_in)]
        got, _ = g.eval(inp)
        assert got == po.evaluate(nodes, inp, wit, "circom")
    return g


@pytest.mark.parametrize("n_regs", [4, 5, 8, 24, 64])
def test_random_graphs_all_ops(n_regs):
    rnd = random.Random(100 + n_regs)
    for _ in range(25):
        nodes, wit, imap = util.random_graph(rnd, n_ops=250)
        g = _check(nodes, wit, imap, n_regs, rnd)
        if n_regs <= 5:
            assert g.info["spill_st"] > 0          # tiny register files must spill, and still be exact


def test_edge_graphs():
    rnd = random.Random(5)
    # empty witness / constants only / inputs only / duplicated witness entries / dead nodes
    _check([(po.K_INPUT, 0)], [], {}, 8, rnd, n_in=0)
    _check([(po.K_INPUT, 0), (po.K_CONST, 7)], [1, 1, 0, 1], {}, 8, rnd, n_in=0)
    nodes = [(po.K_INPUT, i) for i in range(7)] + [(po.K_DUO, 0, 1, 2), (po.K_DUO, 2, 7, 7), (po.K_DUO, 0, 3, 3)]
    _check(nodes, [0, 8, 8, 3, 3, 7, 1], {"x": (1, 6)}, 8, rnd)
    # TernCond that is itself a witness signal, with constant operands
    nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, 5), (po.K_CONST, 9), (po.K_TRES, 0, 1, 2, 3), (po.K_TRES, 0, 2, 1, 4)]
    _check(nodes, [0, 4, 5, 4], {"x": (1, 1)}, 4, rnd, n_in=1)
    # an input index gap (tree_shake removes unused inputs, SURVEY appendix A)
    nodes = [(po.K_INPUT, 0), (po.K_INPUT, 3), (po.K_DUO, 2, 1, 1)]
    g = util.SimGraph(po.serialize_graph(nodes, [0, 2], {"x": (1, 3)}), 8)
    assert g.info["I"] == 4 and g.eval([1, 0, 0, 21])[0] == [1, 42]


def test_register_pressure_chain():
    """a wide fan-in followed by uses in reverse order defeats any small register file"""
    rnd = random.Random(9)
    nodes = [(po.K_INPUT, i) for i in range(7)]
    first = len(nodes)
    for k in range(60):
        nodes.append((po.K_DUO, 0, 1 + k % 6, 1 + (k + 1) % 6))
    acc = first
    for k in range(59, -1, -1):
        nodes.append((po.K_DUO, 2, acc, first + k))
        acc = len(nodes) - 1
    g = _check(nodes, [0, acc], {"x": (1, 6)}, 6, rnd)
    assert g.info["n_spill"] >= 40


@pytest.mark.parametrize("name,n_regs", [("circuit5_poseidon", 8), ("circuit6_num2bits", 24), ("circuit11_key_expansion", 16),
                                         ("circuit8_sha256_512", 24), ("circuit9_authV2", 24), ("circuit9_authV2", 12)])
def test_golden_circuits(name, n_regs):
    data = util.golden_graph(name)
    g = util.SimGraph(data, n_regs)
    got, st = g.eval(g.inputs_from_json(util.golden_inputs(name)))
    assert st == 0 and po.wtns_from_witness(got) == util.golden_wtns(name)
    man = util.manifest()[name]
    assert g.info["W"] == man["n_witness"] and g.info["I"] == man["n_inputs"] and g.info["n_nodes"] == man["n_nodes"]


def _lc_graph(rnd, n_ops=300, n_inputs=6):
    """Graphs dominated by the patterns the plan compiler rewrites: Mul(value, const) feeding Add/Sub trees
    (-> OP_DOT) and Div nodes (-> batched inversion), with extreme constants / values."""
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]
    consts = []
    for v in [0, 1, 2, po.M - 1, po.M - 2, (po.M >> 1), 1 << 253] + [util.random_value(rnd) for _ in range(10)]:
        consts.append(len(nodes))
        nodes.append((po.K_CONST, v % po.M))
    vals = list(range(1, n_inputs + 1))
    for _ in range(n_ops):
        n = len(nodes)
        r = rnd.random()
        pick = lambda: rnd.choice(vals[-12:]) if rnd.random() < 0.7 else rnd.choice(vals)
        if r < 0.35:
            nodes.append((po.K_DUO, po.DUO["Mul"], pick(), rnd.choice(consts)) if rnd.random() < 0.5
                         else (po.K_DUO, po.DUO["Mul"], rnd.choice(consts), pick()))
        elif r < 0.75:
            a = pick() if rnd.random() < 0.85 else rnd.choice(consts)
            b = pick() if rnd.random() < 0.85 else rnd.choice(consts)
            nodes.append((po.K_DUO, po.DUO["Add" if rnd.random() < 0.6 else "Sub"], a, b))
        elif r < 0.87:
            a = pick() if rnd.random() < 0.7 else consts[1]
            nodes.append((po.K_DUO, po.DUO["Div"], a, pick()))
        elif r < 0.93:
            nodes.append((po.K_DUO, po.DUO["Mul"], pick(), pick()))
        else:
            nodes.append((po.K_DUO, po.DUO["Sub"], pick(), pick()))         # x - x = 0 now and then: Div by zero below
        vals.append(n)
    n = len(nodes)
    wit = [0] + [rnd.randrange(n) for _ in range(25)] + list(range(n - 8, n))
    return nodes, wit, {"x": (1, n_inputs)}


@pytest.mark.parametrize("n_regs,div_batch", [(6, 2), (12, 8), (16, 3), (32, 16)])
def test_linear_combination_fusion_and_div_batching(n_regs, div_batch):
    rnd = random.Random(7000 + n_regs)
    fused = batched = 0
    for t in range(20):
        nodes, wit, imap = _lc_graph(rnd)
        data = po.serialize_graph(nodes, wit, imap)
        g = util.SimGraph(data, n_regs, fuse=True, div_batch=div_batch)
        plain = util.SimGraph(data, n_regs, fuse=False, div_batch=1)
        assert plain.info["n_dot"] == 0 and plain.info["inversions"] == plain.info["div_nodes"]
        for row in range(4):
            inp = [1] + [rnd.choice([0, 1, po.M - 1, po.M - 2, (1 << 256) - 1]) if rnd.random() < 0.4 else util.random_value(rnd)
                         for _ in range(6)]
            want = po.evaluate(nodes, inp, wit, "circom")
            assert g.eval(inp)[0] == want, (t, row)
            assert plain.eval(inp)[0] == want, (t, row)
        fused += g.info["n_dot"]
        batched += g.info["div_nodes"] - g.info["inversions"]
    assert fused > 0 and batched > 0


def test_dot_worst_case_bounds():
    """every term at its maximum (value M-1, constant M-1 -> largest products) for each term count / kind mix the
    compiler may emit: the reduced sum must stay exact"""
    M = po.M
    for n_mac in range(0, 9):
        for n_plain in range(0, 5):
            if n_mac == 0:
                continue
            nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, M - 1), (po.K_CONST, 1)]
            acc = None
            for _ in range(n_mac):
                nodes.append((po.K_DUO, po.DUO["Mul"], 1, 2))
                m = len(nodes) - 1
                if acc is None:
                    acc = m
                else:
                    nodes.append((po.K_DUO, po.DUO["Add"], acc, m)); acc = len(nodes) - 1
            for k in range(n_plain):
                nodes.append((po.K_DUO, po.DUO["Add" if k % 2 == 0 else "Sub"], acc, 1)); acc = len(nodes) - 1
            wit = [0, acc]
            g = util.SimGraph(po.serialize_graph(nodes, wit, {"x": (1, 1)}), 16)
            for x in (M - 1, 0, 1, M - 2):
                assert g.eval([1, x])[0] == po.evaluate(nodes, [1, x], wit, "circom"), (n_mac, n_plain, x)


def _narrow_graph(rnd, n_ops=300, n_inputs=6):
    """Graphs that live mostly in the plan compiler's narrow domain (isa.h: F_NARROW): bits and small words cut
    out of arbitrary inputs (Shr+Band, Band with a small mask, Shr by >= 192, comparisons), then sums, products,
    negations, selects, bitwise ops and shifts over them -- with ranges that grow until they leave (-2^62, 2^62)
    and fall back to wide instructions, negative intermediates, wide consumers of narrow values (OP_WIDEN) and
    narrow consumers of wide non-negative values."""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]
    consts = {}
    for v in [0, 1, 2, 3, 5, 7, 31, 32, 62, 63, 64, 100, 192, 200, 253, 254, 255, 0xFF, 0xFFFF, 0xFFFFFFFF, (1 << 61) - 1, (1 << 62) - 1,
              1 << 62, (1 << 64) - 1, po.M - 1, po.M - 2, po.M - 5, po.M - (1 << 40), po.M - (1 << 62) + 1, po.M - (1 << 62), (po.M >> 1),
              (po.M >> 1) + 1, 1 << 20, 1 << 31, 1 << 40] + [util.random_value(rnd) for _ in range(4)]:
        consts[v % po.M] = len(nodes)
        nodes.append((po.K_CONST, v % po.M))
    cl = list(consts.values())
    small_c = [consts[v] for v in (0, 1, 2, 3, 5, 7, 31, 0xFF, 0xFFFF, 0xFFFFFFFF, po.M - 1, po.M - 2, po.M - 5)]
    shift_c = [consts[v] for v in (0, 1, 2, 3, 5, 7, 31, 32, 62, 63, 64, 100, 192, 200, 253, 254, 255)]
    wide = list(range(1, n_inputs + 1))
    narrow = []
    for _ in range(n_ops):
        n = len(nodes)
        r = rnd.random()
        pn = lambda: (rnd.choice(narrow[-10:]) if rnd.random() < 0.6 else rnd.choice(narrow)) if narrow and rnd.random() < 0.9 else rnd.choice(small_c)
        pw = lambda: rnd.choice(wide[-8:]) if rnd.random() < 0.6 else rnd.choice(wide)
        if r < 0.12 or not narrow:     # sources of narrow values
            k = rnd.random()
            if k < 0.4:
                nodes.append((po.K_DUO, D["Shr"], pw(), rnd.choice(shift_c)))
                nodes.append((po.K_DUO, D["Band"], n, rnd.choice([consts[1], consts[0xFF], consts[0xFFFF], consts[0xFFFFFFFF], consts[(1 << 61) - 1]])))
                n += 1
            elif k < 0.55:
                nodes.append((po.K_DUO, D["Band"], rnd.choice([consts[0xFFFF], consts[(1 << 62) - 1], consts[1 << 62], consts[7]]), pw()))
            elif k < 0.7:
                nodes.append((po.K_DUO, D["Shr"], pw(), rnd.choice([consts[192], consts[200], consts[253], consts[254], consts[255], consts[100]])))
            else:
                nodes.append((po.K_DUO, rnd.choice([D["Eq"], D["Neq"], D["Lt"], D["Gt"], D["Leq"], D["Geq"], D["Land"], D["Lor"]]), pw(), pw()))
            narrow.append(n)
        elif r < 0.50:
            nodes.append((po.K_DUO, D["Add" if rnd.random() < 0.55 else "Sub"], pn(), pn())); narrow.append(n)
        elif r < 0.62:
            nodes.append((po.K_DUO, D["Mul"], pn(), pn() if rnd.random() < 0.6 else rnd.choice(small_c + [consts[1 << 20], consts[1 << 31], consts[1 << 40]]))); narrow.append(n)
        elif r < 0.66:
            nodes.append((po.K_UNO, 0, pn())); narrow.append(n)
        elif r < 0.72:
            nodes.append((po.K_TRES, 0, pn() if rnd.random() < 0.7 else pw(), pn(), pn())); narrow.append(n)
        elif r < 0.80:
            nodes.append((po.K_DUO, rnd.choice([D["Band"], D["Bor"], D["Bxor"]]), pn(), pn())); narrow.append(n)
        elif r < 0.86:
            op = rnd.choice([D["Shr"], D["Shl"]])
            nodes.append((po.K_DUO, op, pn(), rnd.choice(shift_c[:10]) if rnd.random() < 0.8 else pn())); narrow.append(n)
        elif r < 0.92:
            nodes.append((po.K_DUO, rnd.choice([D["Eq"], D["Neq"], D["Lt"], D["Gt"], D["Leq"], D["Geq"], D["Land"], D["Lor"]]), pn(), pn())); narrow.append(n)
        else:                          # wide consumers of narrow values, results are wide values again
            op = rnd.choice([D["Mul"], D["Add"], D["Sub"], D["Div"], D["Band"], D["Bxor"], D["Lt"], D["Idiv"], D["Mod"], D["Shr"]])
            a, b = (pn(), pw()) if rnd.random() < 0.5 else (pw(), pn())
            if rnd.random() < 0.2:
                b = rnd.choice(cl)
            nodes.append((po.K_DUO, op, a, b)); wide.append(n)
    n = len(nodes)
    wit = [0] + [rnd.randrange(n) for _ in range(40)] + list(range(n - 10, n))
    return nodes, wit, {"x": (1, n_inputs)}


@pytest.mark.parametrize("n_regs,fuse", [(4, True), (6, True), (12, True), (12, False), (32, True)])
def test_narrow_typing(n_regs, fuse):
    rnd = random.Random(9100 + n_regs + int(fuse))
    n_narrow = n_widen = 0
    for t in range(30):
        nodes, wit, imap = _narrow_graph(rnd)
        data = po.serialize_graph(nodes, wit, imap)
        g = util.SimGraph(data, n_regs, fuse=fuse)
        off = util.SimGraph(data, n_regs, fuse=fuse, narrow=False)
        assert off.info["narrow_instrs"] == 0 and off.info["widen"] == 0
        for row in range(4):
            inp = [1] + [rnd.choice([0, 1, po.M - 1, po.M - 2, (1 << 256) - 1, (1 << 62) - 1, 1 << 62, (1 << 64) - 1]) if rnd.random() < 0.3
                         else util.random_value(rnd) for _ in range(6)]
            want = po.evaluate(nodes, inp, wit, "circom")
            assert g.eval(inp)[0] == want, (t, row)
            assert off.eval(inp)[0] == want, (t, row)
        n_narrow += g.info["narrow_instrs"]
        n_widen += g.info["widen"]
    assert n_narrow > 1000 and n_widen > 0


def test_narrow_range_limits():
    """sums and products right at the +-2^62 boundary of the narrow domain, and negative results as witness values"""
    M = po.M
    D = po.DUO
    for bits in (30, 31, 32, 40, 61, 62):
        mask = (1 << bits) - 1
        nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_INPUT, 2), (po.K_CONST, mask), (po.K_CONST, 0), (po.K_CONST, 1)]
        nodes.append((po.K_DUO, D["Band"], 1, 3)); a = 6
        nodes.append((po.K_DUO, D["Band"], 2, 3)); b = 7
        nodes += [(po.K_DUO, D["Mul"], a, b), (po.K_DUO, D["Sub"], 4, a), (po.K_DUO, D["Sub"], b, a), (po.K_DUO, D["Mul"], 9, b),
                  (po.K_DUO, D["Add"], a, b), (po.K_DUO, D["Add"], 12, 12), (po.K_DUO, D["Mul"], 10, 10), (po.K_UNO, 0, 8),
                  (po.K_DUO, D["Lt"], 9, 10), (po.K_DUO, D["Geq"], 10, 4), (po.K_TRES, 0, 10, 9, 13), (po.K_DUO, D["Sub"], 18, 5)]
        wit = list(range(len(nodes)))
        g = util.SimGraph(po.serialize_graph(nodes, wit, {"x": (1, 2)}), 8)
        assert g.info["narrow_instrs"] > 0
        for x, y in [(mask, mask), (0, mask), (mask, 0), (0, 0), (1, mask), (M - 1, M - 2), ((1 << 256) - 1, 12345), (mask + 1, mask >> 1)]:
            assert g.eval([1, x, y])[0] == po.evaluate(nodes, [1, x, y], wit, "circom"), (bits, x, y)


def test_pow5_sbox_fusion():
    """Sqr -> Sqr -> Mul(., x) chains (Poseidon S-box) become one OP_POW5 when the intermediates have a single reader and
    their witness positions are encodable; every other shape stays three instructions.  Values are bit-exact either way."""
    rnd = random.Random(55)
    base = [(po.K_INPUT, i) for i in range(3)]
    a, b, c = 3, 4, 5
    sbox = [(po.K_DUO, 0, 1, 1), (po.K_DUO, 0, a, a), (po.K_DUO, 0, b, 1)]          # x = input 1
    cases = [
        (sbox, [0, a, b, c], 1),                 # in2, in4, out consecutive: fused
        (sbox, [0, a, c, b], 1),                 # a^4 after a^5: delta 2, fused
        (sbox, [0, c, b, a], 0),                 # a^4 before a^2: not encodable
        (sbox, [0, c], 1),                       # intermediates are not witness signals
        (sbox, [0, a, c], 1),
        (sbox, [0, b, c], 0),                    # a^4 stored but a^2 not: not encodable
        (sbox, [0, a, a, b, c], 0),              # a^2 at two positions
        (sbox + [(po.K_DUO, 2, a, 2)], [0, a, b, c, 6], 0),          # a^2 has a second reader
        (sbox + [(po.K_DUO, 2, b, 2)], [0, a, b, c, 6], 0),          # a^4 has a second reader
        ([(po.K_DUO, 0, 1, 1), (po.K_DUO, 0, a, a), (po.K_DUO, 0, b, 2)], [0, a, b, c], 0),   # last factor is not x
        ([(po.K_DUO, 0, 1, 1), (po.K_DUO, 0, a, a), (po.K_DUO, 0, 1, b)], [0, a, b, c], 1),   # operands swapped
    ]
    for extra, wit, want_fused in cases:
        nodes = base + extra
        g = util.SimGraph(po.serialize_graph(nodes, wit, {"x": (1, 2)}), 8)
        assert g.info["pow5"] == want_fused, (wit, extra)
        g0 = util.SimGraph(po.serialize_graph(nodes, wit, {"x": (1, 2)}), 8, pow5=False)
        assert g0.info["pow5"] == 0
        for _ in range(3):
            inp = [1, util.random_value(rnd), rnd.randrange(1 << 256)]
            want = po.evaluate(nodes, inp, wit, "circom")
            assert g.eval(inp)[0] == want and g0.eval(inp)[0] == want
    # the golden Poseidon graphs are where it matters
    for name, n in (("circuit5_poseidon", 71), ("poseidon2", None)):
        g = util.SimGraph(util.golden_graph(name), 12)
        assert g.info["pow5"] == n if n is not None else g.info["pow5"] > 0


def test_poseidon_like_graphs():
    """random graphs with Poseidon's shapes through the throughput plan: S-box fusion in every operand / witness order"""
    fused = 0
    for seed in range(150):
        rnd = random.Random(4000 + seed)
        nodes, wit, imap = util.poseidon_like_graph(rnd, rnd.choice([2, 3, 5]), rnd.choice([3, 8, 20]))
        g = _check(nodes, wit, imap, rnd.choice([6, 8, 12, 24]), rnd, n_rows=2)
        fused += g.info["pow5"]
    assert fused > 100


def matrix_corpus():
    """The corpus of the plan-option matrix (here on the simulator, tests/test_gpu_plan_matrix.py on the GPU):
    [(name, nodes, witness, input map, rows)].  DOT ladder (1..16 terms at every ring offset, worst-case operands),
    Div groups of 1..16 with their zero patterns, the narrow range limits, a constant-heavy graph, and random, linear-
    combination, narrow and Poseidon-like graphs."""
    M = po.M
    out = []
    rnd = random.Random(2024)
    for t in range(1, 17):
        nodes, wit, imap = util.dot_ladder_graph(t)
        rows = [[1] + [M - 1] * 6, [1] + [0] * 6, [1] + [(1 << 256) - 1] * 6] + [util.matrix_row(rnd, 6) for _ in range(3)]
        out.append((f"dot_ladder_{t}", nodes, wit, imap, rows))
    for k in range(1, 17):
        nodes, wit, imap = util.div_group_graph(k)
        out.append((f"div_group_{k}", nodes, wit, imap, util.div_group_rows(k, rnd)))
    for bits, nodes, wit, imap in util.narrow_limit_graphs():
        vals = util.narrow_limit_values(bits)
        out.append((f"narrow_limits_{bits}", nodes, wit, imap, [[1, x, y] for x in vals for y in vals]))
    nodes, wit, imap = util.const_heavy_graph(rnd)
    out.append(("const_heavy", nodes, wit, imap, [util.matrix_row(rnd, 6) for _ in range(6)] + [[1] + [M - 1] * 6]))
    for k in range(2):
        for name, gen in (("random", lambda: util.random_graph(rnd, n_ops=400)), ("lc", lambda: _lc_graph(rnd)),
                          ("narrow", lambda: _narrow_graph(rnd)), ("poseidon", lambda: util.poseidon_like_graph(rnd, 3, 8))):
            nodes, wit, imap = gen()
            out.append((f"{name}_{k}", nodes, wit, imap, [util.matrix_row(rnd, 6) for _ in range(6)]))
    return out


_PLAN_ONLY = {}
for _name, _env in util.PLAN_VARIANTS:           # the variants that change the compiled program (the others are launch options)
    _PLAN_ONLY.setdefault(tuple(sorted(util.sim_options(_env).items())), _name)


@pytest.mark.parametrize("variant", sorted(_PLAN_ONLY.values()))
def test_plan_matrix_corpus(variant):
    """every corpus graph under every plan option of the matrix, on the simulator, against the C oracle; and the corpus
    reaches what it is there for (util.assert_plan_coverage)"""
    from oracle import cref
    env = dict(util.PLAN_VARIANTS)[variant]
    opts = util.sim_options(env)
    cov = None
    for name, nodes, wit, imap, rows in matrix_corpus():
        data = po.serialize_graph(nodes, wit, imap)
        g = util.SimGraph(data, **opts)
        want = cref.CGraph(data).evaluate_batch(np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32), 4)
        for b, r in enumerate(rows):
            assert g.eval(r)[0] == util.unpack_u256(want[b].tobytes()), (name, b)
        c = util.plan_coverage(g.code())
        cov = c if cov is None else util.merge_coverage(cov, c)
    util.assert_plan_coverage(cov, util.VARIANT_FEATURES.get(variant, ()))
